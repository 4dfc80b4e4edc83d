// b200sd -- the non-GEMM kernels of the UNet backward pass (autograd.backward through
// UNet2DConditionModel.forward, finetune_sd.py:494; SURVEY.md row A9): gradient cast + bias-gradient column
// sums, GroupNorm(+SiLU) / LayerNorm backward, GEGLU forward/backward for the training path (which keeps the
// pre-activation), the transposes of the two resamplers, and the degenerate 4-channel convs at the UNet ends.
// All are bandwidth-bound passes; parameter gradients are ACCUMULATED into fp32 with atomics (the flat
// gradient buffer is zeroed once per optimizer step), activation gradients are written or accumulated as asked.
#include <atomic>
#include <cmath>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }
// d/dz [z * sigmoid(z)]
__device__ __forceinline__ float silu_grad_f(float z) {
    const float s = sigmoid_f(z);
    return s * (1.0f + z * (1.0f - s));
}
// d/dx [0.5 x (1 + erf(x / sqrt 2))] = Phi(x) + x phi(x)
__device__ __forceinline__ float gelu_erf_grad_f(float x) {
    const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752f));
    const float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
    return cdf + x * pdf;
}

int ew_grid(int64_t total, int threads) {
    int64_t blocks = (total + threads - 1) / threads;
    const int64_t cap = (int64_t)b200sd_num_sms() * 8;
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

// ---- gradient prep: optional bf16 copy (tensor-core operand) + per-column sums (bias gradient) --------------
// grid (ceil(N/64), row slabs); block 256 = 8 column vectors x 32 rows.  A slab never straddles an image when
// rows_per_block divides rows_per_image, so the same kernel produces the per-image sums of the time-embedding
// gradient (colsum + image * ldcs).
template <int DT>
__global__ void __launch_bounds__(256) grad_prep_kernel(const void* __restrict__ in, bf16* __restrict__ out,
                                                        float* __restrict__ colsum, int rows, int N, int ld,
                                                        int rows_per_block, int rows_per_image, int ldcs) {
    __shared__ float s_acc[32][65];
    const int v = threadIdx.x & 7, r = threadIdx.x >> 3;
    const int c = blockIdx.x * 64 + v * 8;
    const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c < N) {
#pragma unroll 4
        for (int row = r0 + r; row < r1; row += 32) {
            float f[8];
            ld8<DT>(in, (size_t)row * ld + c, f);
            if (out) st8<B200SD_BF16>(out, (size_t)row * ld + c, f);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += f[j];
        }
    }
    if (colsum == nullptr) return;
#pragma unroll
    for (int j = 0; j < 8; ++j) s_acc[r][v * 8 + j] = acc[j];
    __syncthreads();
    if (threadIdx.x < 64 && blockIdx.x * 64 + threadIdx.x < N) {
        float a = 0.f;
#pragma unroll 8
        for (int i = 0; i < 32; ++i) a += s_acc[i][threadIdx.x];
        const int img = rows_per_image > 0 ? r0 / rows_per_image : 0;
        atomicAdd(colsum + (size_t)img * ldcs + blockIdx.x * 64 + threadIdx.x, a);
    }
}

// ---- GroupNorm (+SiLU) backward ----------------------------------------------------------------------------
// y = act(gamma * xhat + beta), xhat = (x - mean) * rstd over (pixels x channels-of-group) of one image.
//   g     = dy * act'(z)
//   dx    = rstd * (g gamma - mean_grp(g gamma) - xhat * mean_grp(g gamma xhat))
//   dgamma = sum g xhat,  dbeta = sum g
// Pass 1 (grid groups x batch): recompute mean / rstd of the group, then the two group means and the
// per-channel affine gradients.  Pass 2: elementwise dx (+ optional fp32 addend: the residual path).
template <int DT>
__global__ void __launch_bounds__(512) gn_bwd_stats_kernel(const void* __restrict__ x0, const void* __restrict__ x1, int C0,
                                                           int C1, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, const bf16* __restrict__ dy,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                           float4* __restrict__ stats, int hw, int groups, float eps,
                                                           int silu) {
    extern __shared__ float s_red[];   // [4][blockDim.x]
    __shared__ float s_ms[4];
    const int C = C0 + C1, cpg = C / groups;
    const int g = blockIdx.x, b = blockIdx.y;
    const int rpp = blockDim.x / cpg;           // pixel rows per pass
    const int ch = threadIdx.x % cpg, prow = threadIdx.x / cpg;
    const bool active = prow < rpp;
    const int c = g * cpg + ch;
    const float* xf = nullptr;
    const bf16* xb = nullptr;
    size_t off;
    int pitch;
    {
        const void* src;
        if (c < C0) { src = x0; off = (size_t)b * hw * C0 + c; pitch = C0; }
        else { src = x1; off = (size_t)b * hw * C1 + (c - C0); pitch = C1; }
        if constexpr (DT == B200SD_F32) xf = static_cast<const float*>(src);
        else xb = static_cast<const bf16*>(src);
    }
    auto ldx = [&](int p) -> float {
        if constexpr (DT == B200SD_F32) return __ldg(xf + off + (size_t)p * pitch);
        else return __bfloat162float(xb[off + (size_t)p * pitch]);
    };
    auto block_sum4 = [&](float a0, float a1, float a2, float a3) {
        const int n = blockDim.x;
        s_red[threadIdx.x] = a0; s_red[n + threadIdx.x] = a1; s_red[2 * n + threadIdx.x] = a2; s_red[3 * n + threadIdx.x] = a3;
        __syncthreads();
        if (threadIdx.x < 128) {   // 4 quantities x 32 lanes, fixed order
            const int q = threadIdx.x >> 5, lane = threadIdx.x & 31;
            float a = 0.f;
            for (int i = lane; i < n; i += 32) a += s_red[q * n + i];
            a = warp_sum(a);
            if (lane == 0) s_ms[q] = a;
        }
        __syncthreads();
    };
    // ---- mean / rstd ----
    float s = 0.f, ss = 0.f;
    if (active)
        for (int p = prow; p < hw; p += rpp) { const float v = ldx(p); s += v; ss += v * v; }
    block_sum4(s, ss, 0.f, 0.f);
    const float cnt = (float)hw * (float)cpg;
    const float mean = s_ms[0] / cnt;
    float var = s_ms[1] / cnt - mean * mean;
    if (var < 0.f) var = 0.f;
    const float rstd = rsqrtf(var + eps);
    __syncthreads();
    // ---- group means of (g gamma) and (g gamma xhat); per-channel affine gradients ----
    float a1 = 0.f, a2 = 0.f, dg = 0.f, db = 0.f;
    if (active) {
        const float gm = __ldg(gamma + c), bt = __ldg(beta + c);
        const bf16* dyp = dy + (size_t)b * hw * C + c;
        for (int p = prow; p < hw; p += rpp) {
            const float xh = (ldx(p) - mean) * rstd;
            float gy = __bfloat162float(dyp[(size_t)p * C]);
            if (silu) gy *= silu_grad_f(gm * xh + bt);
            a1 += gy * gm;
            a2 += gy * gm * xh;
            dg += gy * xh;
            db += gy;
        }
    }
    block_sum4(a1, a2, 0.f, 0.f);
    if (threadIdx.x == 0) stats[(size_t)b * groups + g] = make_float4(mean, rstd, s_ms[0] / cnt, s_ms[1] / cnt);
    if (dgamma != nullptr) {
        __syncthreads();
        s_red[threadIdx.x] = dg;
        s_red[blockDim.x + threadIdx.x] = db;
        __syncthreads();
        if (threadIdx.x < cpg) {
            float tg = 0.f, tb = 0.f;
            for (int r = 0; r < rpp; ++r) { tg += s_red[r * cpg + threadIdx.x]; tb += s_red[blockDim.x + r * cpg + threadIdx.x]; }
            atomicAdd(dgamma + g * cpg + threadIdx.x, tg);
            atomicAdd(dbeta + g * cpg + threadIdx.x, tb);
        }
    }
}


// ---- fast path of the GroupNorm backward statistics (forward kept mean / rstd) --------------------------------------
// Because gamma is constant per channel, the two group means are sums over the group's channels of
//   gamma_c * sum_p g        and        gamma_c * sum_p g xhat,
// i.e. exactly the per-channel dbeta_c / dgamma_c.  Pass 1 therefore only needs the per-channel pixel sums: every thread
// owns ONE 8-channel vector and walks down its pixel slab with 16 / 32-byte loads (grid: slabs x channel chunks x batch),
// the block folds its rows in smem and adds 2 floats per channel to a small workspace.  Pass 2 (one block per image)
// turns them into the group means, accumulates dgamma / dbeta and re-zeroes the workspace.
template <int DT>
__global__ void __launch_bounds__(256) gn_bwd_partial_kernel(const void* __restrict__ x0, const void* __restrict__ x1, int C0, int C1,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             const bf16* __restrict__ dy, const float* __restrict__ mean_rstd,
                                                             float* __restrict__ chan_ws, int hw, int groups, int silu, int VC,
                                                             int pix_per_slab) {
    extern __shared__ float s_fold[];   // [2][R][VC * 8]
    const int C = C0 + C1, cpg = C / groups, C8 = C / 8;
    const int b = blockIdx.z, chunk = blockIdx.y;
    const int R = blockDim.x / VC;
    const int vec = threadIdx.x % VC, prow = threadIdx.x / VC;
    const int v8 = chunk * VC + vec;
    const int c = v8 * 8;
    const bool active = prow < R && v8 < C8;
    float sg[8], sx[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sg[j] = 0.f; sx[j] = 0.f; }
    if (active) {
        float gm[8], bt[8], mu[8], rs[8];
        ld8<B200SD_F32>(gamma, c, gm);
        ld8<B200SD_F32>(beta, c, bt);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int g = (c + j) / cpg;
            mu[j] = __ldg(mean_rstd + ((size_t)b * groups + g) * 2);
            rs[j] = __ldg(mean_rstd + ((size_t)b * groups + g) * 2 + 1);
        }
        const void* src;
        size_t off;
        int pitch;
        if (c < C0) { src = x0; off = (size_t)b * hw * C0 + c; pitch = C0; }
        else { src = x1; off = (size_t)b * hw * C1 + (c - C0); pitch = C1; }
        const int p0 = blockIdx.x * pix_per_slab, p1 = min(hw, p0 + pix_per_slab);
#pragma unroll 2
        for (int p = p0 + prow; p < p1; p += R) {
            float f[8], g[8];
            ld8<DT>(src, off + (size_t)p * pitch, f);
            ld8<B200SD_BF16>(dy, ((size_t)b * hw + p) * C + c, g);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float xh = (f[j] - mu[j]) * rs[j];
                float gy = g[j];
                if (silu) gy *= silu_grad_f(gm[j] * xh + bt[j]);
                sg[j] += gy;
                sx[j] += gy * xh;
            }
        }
    }
    const int W = VC * 8;
    if (prow < R) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            s_fold[(size_t)prow * W + vec * 8 + j] = sg[j];
            s_fold[(size_t)(R + prow) * W + vec * 8 + j] = sx[j];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * W; i += blockDim.x) {
        const int which = i / W, col = i % W;
        const int ch = chunk * W + col;
        if (ch >= C) continue;
        float a = 0.f;
        for (int r = 0; r < R; ++r) a += s_fold[(size_t)(which * R + r) * W + col];
        chan_ws[(((size_t)b * gridDim.x + blockIdx.x) * C + ch) * 2 + which] = a;   // this slab's partial (no atomics: deterministic)
    }
}

// grid (groups, batch): one block folds the slab partials of its group's channels in a fixed order
__global__ void __launch_bounds__(256) gn_bwd_finalize_kernel(const float* __restrict__ gamma, const float* __restrict__ mean_rstd,
                                                              const float* __restrict__ chan_ws, float4* __restrict__ stats,
                                                              float* __restrict__ dgamma, float* __restrict__ dbeta, int C, int hw,
                                                              int groups, int slabs) {
    extern __shared__ float s_part[];   // [parts][2 * cpg] then [2 * cpg] folded
    const int g = blockIdx.x, b = blockIdx.y, cpg = C / groups;
    const int nE = 2 * cpg;                               // (sum g, sum g xhat) per channel of the group, interleaved
    const int parts = max(1, (int)blockDim.x / nE);
    const float* ws = chan_ws + ((size_t)b * slabs * C + (size_t)g * cpg) * 2;
    for (int t = threadIdx.x; t < parts * nE; t += blockDim.x) {
        const int e = t % nE, part = t / nE;
        float a = 0.f;
        for (int sl = part; sl < slabs; sl += parts) a += ws[(size_t)sl * C * 2 + e];
        s_part[part * nE + e] = a;
    }
    __syncthreads();
    float* s_ch = s_part + parts * nE;
    for (int e = threadIdx.x; e < nE; e += blockDim.x) {
        float a = 0.f;
        for (int part = 0; part < parts; ++part) a += s_part[part * nE + e];
        s_ch[e] = a;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s1 = 0.f, s2 = 0.f;
        for (int j = 0; j < cpg; ++j) {
            const float gm = __ldg(gamma + g * cpg + j);
            s1 += gm * s_ch[2 * j];
            s2 += gm * s_ch[2 * j + 1];
        }
        const float inv = 1.0f / ((float)hw * (float)cpg);
        stats[(size_t)b * groups + g] = make_float4(mean_rstd[((size_t)b * groups + g) * 2], mean_rstd[((size_t)b * groups + g) * 2 + 1],
                                                    s1 * inv, s2 * inv);
    }
    if (dgamma != nullptr)
        for (int j = threadIdx.x; j < cpg; j += blockDim.x) {
            atomicAdd(dbeta + g * cpg + j, s_ch[2 * j]);
            atomicAdd(dgamma + g * cpg + j, s_ch[2 * j + 1]);
        }
}

template <int DT, int ODT>
__global__ void __launch_bounds__(256) gn_bwd_apply_kernel(const void* __restrict__ x0, const void* __restrict__ x1, int C0,
                                                           int C1, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, const bf16* __restrict__ dy,
                                                           const float* __restrict__ add_src, void* __restrict__ out0,
                                                           void* __restrict__ out1, int acc0, int acc1,
                                                           const float4* __restrict__ stats, int hw, int groups, int silu,
                                                           int pix_per_block) {
    __shared__ float4 s_st[32];
    const int C = C0 + C1, cpg = C / groups, b = blockIdx.y;
    if (threadIdx.x < groups) s_st[threadIdx.x] = stats[(size_t)b * groups + threadIdx.x];
    __syncthreads();
    const int vpp = C / 8;
    const int p_begin = blockIdx.x * pix_per_block, p_end = min(p_begin + pix_per_block, hw);
    const int total = (p_end - p_begin) * vpp;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int p = p_begin + i / vpp;
        const int c = (i % vpp) * 8;
        const size_t row = (size_t)b * hw + p;
        float f[8], gy[8], gm[8], bt[8], o[8];
        if (c < C0) ld8<DT>(x0, row * C0 + c, f);
        else ld8<DT>(x1, row * C1 + (c - C0), f);
        ld8<B200SD_BF16>(dy, row * C + c, gy);
        ld8<B200SD_F32>(gamma, c, gm);
        ld8<B200SD_F32>(beta, c, bt);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 st = s_st[(c + j) / cpg];
            const float xh = (f[j] - st.x) * st.y;
            float g = gy[j];
            if (silu) g *= silu_grad_f(gm[j] * xh + bt[j]);
            o[j] = st.y * (g * gm[j] - st.z - xh * st.w);
        }
        if (add_src) {
            float a[8];
            ld8<B200SD_F32>(add_src, row * C + c, a);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] += a[j];
        }
        void* dst;
        size_t di;
        int acc;
        if (c < C0) { dst = out0; di = row * C0 + c; acc = acc0; }
        else { dst = out1; di = row * C1 + (c - C0); acc = acc1; }
        if (acc) {
            float t[8];
            ld8<ODT>(dst, di, t);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] += t[j];
        }
        st8<ODT>(dst, di, o);
    }
}

// ---- LayerNorm backward: one warp per row (row in registers), affine gradients reduced per block ------------
template <int P, int DT>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const void* __restrict__ x, const float* __restrict__ gamma,
                                                            const bf16* __restrict__ dy, float* __restrict__ dres,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta, int rows,
                                                            int C, float eps, int rows_per_block) {
    extern __shared__ float s_buf[];   // [8][C]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r_begin = blockIdx.x * rows_per_block, r_end = min(rows, r_begin + rows_per_block);
    float2 dg[P], db[P], gm[P];
#pragma unroll
    for (int i = 0; i < P; ++i) {
        dg[i] = make_float2(0.f, 0.f);
        db[i] = make_float2(0.f, 0.f);
        gm[i] = __ldg(reinterpret_cast<const float2*>(gamma) + lane + 32 * i);
    }
    const float invC = 1.0f / (float)C;
    for (int row = r_begin + warp; row < r_end; row += 8) {
        float2 v[P], g[P];
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < P; ++i) {
            if constexpr (DT == B200SD_F32)
                v[i] = __ldg(reinterpret_cast<const float2*>(static_cast<const float*>(x) + (size_t)row * C) + lane + 32 * i);
            else
                v[i] = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(static_cast<const bf16*>(x) + (size_t)row * C) + lane + 32 * i));
            g[i] = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(dy + (size_t)row * C) + lane + 32 * i));
            s += v[i].x + v[i].y;
        }
        const float mean = warp_sum(s) * invC;
        float ss = 0.f;
#pragma unroll
        for (int i = 0; i < P; ++i) {
            v[i].x -= mean; v[i].y -= mean;
            ss += v[i].x * v[i].x + v[i].y * v[i].y;
        }
        const float rstd = rsqrtf(warp_sum(ss) * invC + eps);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < P; ++i) {
            v[i].x *= rstd; v[i].y *= rstd;                       // xhat
            dg[i].x += g[i].x * v[i].x; dg[i].y += g[i].y * v[i].y;
            db[i].x += g[i].x; db[i].y += g[i].y;
            g[i].x *= gm[i].x; g[i].y *= gm[i].y;                 // dy * gamma
            s1 += g[i].x + g[i].y;
            s2 += g[i].x * v[i].x + g[i].y * v[i].y;
        }
        s1 = warp_sum(s1) * invC;
        s2 = warp_sum(s2) * invC;
        float2* dst = reinterpret_cast<float2*>(dres + (size_t)row * C);
#pragma unroll
        for (int i = 0; i < P; ++i) {
            float2 o = dst[lane + 32 * i];
            o.x += rstd * (g[i].x - s1 - v[i].x * s2);
            o.y += rstd * (g[i].y - s1 - v[i].y * s2);
            dst[lane + 32 * i] = o;
        }
    }
    if (dgamma == nullptr) return;
    for (int pass = 0; pass < 2; ++pass) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < P; ++i)
            reinterpret_cast<float2*>(s_buf + (size_t)warp * C)[lane + 32 * i] = pass == 0 ? dg[i] : db[i];
        __syncthreads();
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            float a = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) a += s_buf[(size_t)w * C + c];
            atomicAdd((pass == 0 ? dgamma : dbeta) + c, a);
        }
    }
}

// ---- GEGLU (training path: natural [values | gates] column order, pre-activation kept) ----------------------
__global__ void geglu_fwd_kernel(const bf16* __restrict__ u, bf16* __restrict__ out, int64_t rows, int Ch8) {
    const int64_t total = rows * Ch8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t row = i / Ch8;
        const int c = (int)(i % Ch8) * 8;
        float v[8], g[8], o[8];
        ld8<B200SD_BF16>(u, (size_t)row * Ch8 * 16 + c, v);
        ld8<B200SD_BF16>(u, (size_t)row * Ch8 * 16 + (size_t)Ch8 * 8 + c, g);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = v[j] * gelu_erf_f(g[j]);
        st8<B200SD_BF16>(out, (size_t)row * Ch8 * 8 + c, o);
    }
}
__global__ void geglu_bwd_kernel(const bf16* __restrict__ u, const bf16* __restrict__ dff, bf16* __restrict__ du,
                                 int64_t rows, int Ch8) {
    const int64_t total = rows * Ch8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t row = i / Ch8;
        const int c = (int)(i % Ch8) * 8;
        const size_t iv = (size_t)row * Ch8 * 16 + c, ig = iv + (size_t)Ch8 * 8;
        float v[8], g[8], d[8], dv[8], dgt[8];
        ld8<B200SD_BF16>(u, iv, v);
        ld8<B200SD_BF16>(u, ig, g);
        ld8<B200SD_BF16>(dff, (size_t)row * Ch8 * 8 + c, d);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            dv[j] = d[j] * gelu_erf_f(g[j]);
            dgt[j] = d[j] * v[j] * gelu_erf_grad_f(g[j]);
        }
        st8<B200SD_BF16>(du, iv, dv);
        st8<B200SD_BF16>(du, ig, dgt);
    }
}

// ---- transposes of the resamplers ---------------------------------------------------------------------------
// nearest x2 upsample backward: dx[b,y,x,:] (+)= sum of the 2x2 block of dy
__global__ void upsample2x_bwd_kernel(const bf16* __restrict__ dy, float* __restrict__ dx, int batch, int H, int W, int C8,
                                      int accumulate) {
    const int64_t total = (int64_t)batch * H * W * C8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i % C8);
        int64_t p = i / C8;
        const int x = (int)(p % W);
        p /= W;
        const int y = (int)(p % H);
        const int b = (int)(p / H);
        float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float v[8];
            ld8<B200SD_BF16>(dy, (size_t)(((int64_t)(b * 2 * H + 2 * y + (q >> 1)) * 2 * W + 2 * x + (q & 1)) * C8 + c) * 8, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] += v[j];
        }
        if (accumulate) {
            float t[8];
            ld8<B200SD_F32>(dx, (size_t)i * 8, t);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] += t[j];
        }
        st8<B200SD_F32>(dx, (size_t)i * 8, o);
    }
}
// col2im of the stride-2 pad-1 3x3 im2col: dx[b,y,x,:] (+)= sum over taps (ky,kx) with y = 2 oy + ky - 1, x = 2 ox + kx - 1
__global__ void col2im_s2_kernel(const bf16* __restrict__ dcol, float* __restrict__ dx, int batch, int H, int W, int C8,
                                 int accumulate) {
    const int OH = H / 2, OW = W / 2;
    const int64_t total = (int64_t)batch * H * W * C8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i % C8);
        int64_t p = i / C8;
        const int x = (int)(p % W);
        p /= W;
        const int y = (int)(p % H);
        const int b = (int)(p / H);
        float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int ky = 0; ky < 3; ++ky) {
            const int ty = y + 1 - ky;
            if (ty < 0 || (ty & 1) || (ty >> 1) >= OH) continue;
            for (int kx = 0; kx < 3; ++kx) {
                const int tx = x + 1 - kx;
                if (tx < 0 || (tx & 1) || (tx >> 1) >= OW) continue;
                float v[8];
                ld8<B200SD_BF16>(dcol, (size_t)((((int64_t)(b * OH + (ty >> 1)) * OW + (tx >> 1)) * 9 + ky * 3 + kx) * C8 + c) * 8, v);
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] += v[j];
            }
        }
        if (accumulate) {
            float t[8];
            ld8<B200SD_F32>(dx, (size_t)i * 8, t);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] += t[j];
        }
        st8<B200SD_F32>(dx, (size_t)i * 8, o);
    }
}

// ---- the 4-channel convs at the UNet ends -------------------------------------------------------------------
// conv_out data gradient: dt[p, ci] = sum_tap sum_co dout[b, co, p - d(tap)] * w[co][tap][ci]   (bf16 NHWC out)
__global__ void __launch_bounds__(256) conv_out_dgrad_kernel(const float* __restrict__ dout, const float* __restrict__ w,
                                                             bf16* __restrict__ dt, int batch, int Cin, int Cout, int H, int W) {
    const int C8 = Cin / 8;
    const int64_t total = (int64_t)batch * H * W * C8, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i % C8) * 8;
        int64_t p = i / C8;
        const int x = (int)(p % W);
        p /= W;
        const int y = (int)(p % H);
        const int b = (int)(p / H);
        float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int tap = 0; tap < 9; ++tap) {
            const int yy = y - (tap / 3 - 1), xx = x - (tap % 3 - 1);
            if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
            for (int co = 0; co < Cout; ++co) {
                const float g = __ldg(dout + ((size_t)(b * Cout + co) * H + yy) * W + xx);
                float wv[8];
                ld8<B200SD_F32>(w, (size_t)(co * 9 + tap) * Cin + c, wv);
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] += g * wv[j];
            }
        }
        st8<B200SD_BF16>(dt, (size_t)i * 8, o);
    }
}

// Weight gradient of a conv between a wide NHWC tensor (Cw channels) and a narrow NCHW fp32 tensor (Cn <= 4):
//   acc[cw][tap][cn] = sum_q wide[q, cw] * narrow[b, cn, q + sign * d(tap)]
// conv_in  (wide = dy,  sign = +1): dW[co = cw][tap][ci = cn]   -> out_mode 0: dw[(cw * 9 + tap) * Cn + cn]
// conv_out (wide = act, sign = -1): dW[co = cn][tap][ci = cw]   -> out_mode 1: dw[(cn * 9 + tap) * Cw + cw]
template <int DT>
__global__ void __launch_bounds__(256) conv_small_wgrad_kernel(const void* __restrict__ wide, const float* __restrict__ narrow,
                                                               float* __restrict__ dw, int batch, int H, int W, int Cw, int Cn,
                                                               int sign, int out_mode, int pix_per_block) {
    const int cw = blockIdx.y * blockDim.x + threadIdx.x;
    const int hw = H * W, total = batch * hw;
    const int q0 = blockIdx.x * pix_per_block, q1 = min(total, q0 + pix_per_block);
    float acc[9][4];
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int n = 0; n < 4; ++n) acc[t][n] = 0.f;
    for (int q = q0; q < q1; ++q) {
        const int b = q / hw, rem = q % hw, y = rem / W, x = rem % W;
        float wv = 0.f;
        if (cw < Cw) {
            if constexpr (DT == B200SD_F32) wv = __ldg(static_cast<const float*>(wide) + (size_t)q * Cw + cw);
            else wv = __bfloat162float(static_cast<const bf16*>(wide)[(size_t)q * Cw + cw]);
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int yy = y + sign * (t / 3 - 1), xx = x + sign * (t % 3 - 1);
            if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
#pragma unroll
            for (int n = 0; n < 4; ++n)
                if (n < Cn) acc[t][n] += wv * __ldg(narrow + ((size_t)(b * Cn + n) * H + yy) * W + xx);
        }
    }
    if (cw >= Cw) return;
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int n = 0; n < 4; ++n)
            if (n < Cn) atomicAdd(dw + (out_mode == 0 ? ((size_t)(cw * 9 + t) * Cn + n) : ((size_t)(n * 9 + t) * Cw + cw)), acc[t][n]);
}

// per-channel sum of an NCHW fp32 tensor (bias gradient of conv_out): grid (C), accumulated
__global__ void __launch_bounds__(256) nchw_channel_sum_kernel(const float* __restrict__ x, float* __restrict__ out, int batch,
                                                               int C, int hw) {
    __shared__ float s_w[8];
    const int c = blockIdx.x;
    float a = 0.f;
    for (int i = threadIdx.x; i < batch * hw; i += blockDim.x) a += x[((size_t)(i / hw) * C + c) * hw + i % hw];
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += s_w[i];
        atomicAdd(out + c, t);
    }
}

// ---- small elementwise helpers of the time-embedding backward -----------------------------------------------
__global__ void cast_act_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t n, int silu) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float v = in[i];
        if (silu) v = v * sigmoid_f(v);
        out[i] = __float2bfloat16(v);
    }
}
__global__ void silu_bwd_mul_kernel(const float* __restrict__ pre, float* __restrict__ g, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        g[i] *= silu_grad_f(pre[i]);
}

// ---- flat-buffer kernels of the optimizer step ----------------------------------------------------------------
// fp32 master -> bf16 tensor-core copy, 8 elements per thread
__global__ void cast_flat_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t n8) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        float v[8];
        ld8<B200SD_F32>(in, (size_t)i * 8, v);
        st8<B200SD_BF16>(out, (size_t)i * 8, v);
    }
}

// AdamW (decoupled weight decay, torch.optim.AdamW semantics) over the flat kernel-layout buffers, fused with the
// gradient averaging of data parallelism (grad_scale = 1 / world), the bf16 re-cast of the updated weights and
// (optionally) the zeroing of the gradient buffer for the next step: one pass, 16 B read + 14 B written per parameter.
__global__ void __launch_bounds__(256) adamw_flat_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                         float* __restrict__ v, bf16* __restrict__ wb, int64_t n4, float lr,
                                                         float beta1, float beta2, float eps, float wd, float bc1, float rsqrt_bc2,
                                                         float grad_scale, int zero_grad) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 P = reinterpret_cast<float4*>(p)[i], G = reinterpret_cast<float4*>(g)[i];
        float4 M = reinterpret_cast<float4*>(m)[i], V = reinterpret_cast<float4*>(v)[i];
        float* pp = &P.x; float* gg = &G.x; float* mm = &M.x; float* vv = &V.x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float gr = gg[j] * grad_scale;
            pp[j] *= (1.0f - lr * wd);
            mm[j] = beta1 * mm[j] + (1.0f - beta1) * gr;
            vv[j] = beta2 * vv[j] + (1.0f - beta2) * gr * gr;
            const float denom = sqrtf(vv[j]) * rsqrt_bc2 + eps;
            pp[j] -= (lr / bc1) * (mm[j] / denom);
        }
        reinterpret_cast<float4*>(p)[i] = P;
        reinterpret_cast<float4*>(m)[i] = M;
        reinterpret_cast<float4*>(v)[i] = V;
        if (zero_grad) reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        uint2 u;
        u.x = pack_bf16x2(P.x, P.y);
        u.y = pack_bf16x2(P.z, P.w);
        reinterpret_cast<uint2*>(wb)[i] = u;
    }
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" int b200sd_grad_prep(const void* in, int in_dtype, void* out_bf16, float* colsum, int rows, int N, int ld,
                                int rows_per_image, int ldcs, b200sd_stream_t stream) {
    B200SD_REQUIRE(in != nullptr && (out_bf16 != nullptr || colsum != nullptr), "grad_prep: null pointer");
    B200SD_REQUIRE(rows > 0 && N > 0 && N % 8 == 0 && ld % 8 == 0 && ld >= N, "grad_prep: bad sizes rows=%d N=%d ld=%d", rows, N, ld);
    B200SD_REQUIRE(in_dtype == B200SD_F32 || in_dtype == B200SD_BF16, "grad_prep: bad dtype");
    B200SD_REQUIRE(rows_per_image <= 0 || rows % rows_per_image == 0, "grad_prep: rows must be a multiple of rows_per_image");
    // slab height: enough blocks to fill the machine, a divisor of the image so a slab never straddles images
    const int unit = rows_per_image > 0 ? rows_per_image : rows;
    const int col_blocks = ceil_div(N, 64);
    int rpb = ceil_div(rows, ceil_div(b200sd_num_sms() * 4, col_blocks));
    if (rpb < 32) rpb = 32;
    if (rpb > unit) rpb = unit;
    if (rows_per_image > 0) {
        while (unit % rpb != 0) ++rpb;   // next divisor of the image height (terminates at rpb == unit)
    }
    dim3 grid(col_blocks, ceil_div(rows, rpb));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (in_dtype == B200SD_F32)
        grad_prep_kernel<B200SD_F32><<<grid, dim3(256), 0, s>>>(in, static_cast<bf16*>(out_bf16), colsum, rows, N,
                                  ld, rpb, rows_per_image, ldcs);
    else
        grad_prep_kernel<B200SD_BF16><<<grid, dim3(256), 0, s>>>(in, static_cast<bf16*>(out_bf16), colsum, rows, N,
                                  ld, rpb, rows_per_image, ldcs);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// workspace: [kGnBwdMaxBatch * 32] float4 group statistics, then per-(image, pixel slab) per-channel partial sums
// [batch * slabs][C][2] with batch * slabs <= kGnBwdMaxSlabs + batch.  Plain scratch: no zero-on-entry contract.
constexpr int kGnBwdMaxC = 4096;
constexpr int kGnBwdMaxBatch = 1024;
constexpr int kGnBwdMaxSlabs = 640;
extern "C" int b200sd_groupnorm_bwd_workspace_floats(int batch) {
    return 4 * kGnBwdMaxBatch * 32 + 2 * (kGnBwdMaxSlabs + batch) * kGnBwdMaxC;
}

extern "C" int b200sd_groupnorm_silu_bwd(const void* x0, const void* x1, int C0, int C1, int in_dtype, const float* gamma,
                                         const float* beta, const void* dy, const float* add_src, void* out0, void* out1,
                                         int out_dtype, int accumulate0, int accumulate1, float* dgamma, float* dbeta,
                                         const float* mean_rstd, float* workspace, int batch, int hw, int groups, float eps,
                                         int silu, b200sd_stream_t stream) {
    B200SD_REQUIRE(x0 && gamma && beta && dy && out0 && workspace, "groupnorm_bwd: null pointer");
    if (!x1) C1 = 0;
    B200SD_REQUIRE(C1 == 0 || out1 != nullptr, "groupnorm_bwd: out1 missing for the second source");
    B200SD_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), "groupnorm_bwd: dgamma / dbeta must both be given or both NULL");
    const int C = C0 + C1;
    B200SD_REQUIRE(batch > 0 && batch <= kGnBwdMaxBatch && hw > 0 && groups > 0 && groups <= 32 && C % groups == 0, "groupnorm_bwd: bad sizes");
    B200SD_REQUIRE(C0 % 8 == 0 && C1 % 8 == 0, "groupnorm_bwd: channel counts must be multiples of 8");
    B200SD_REQUIRE(in_dtype == B200SD_BF16 || in_dtype == B200SD_F32, "groupnorm_bwd: bad input dtype");
    B200SD_REQUIRE(out_dtype == B200SD_BF16 || out_dtype == B200SD_F32, "groupnorm_bwd: bad output dtype");
    const int cpg = C / groups;
    B200SD_REQUIRE(cpg <= 512, "groupnorm_bwd: %d channels per group unsupported", cpg);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float4* stats = reinterpret_cast<float4*>(workspace);
    if (mean_rstd != nullptr && C <= kGnBwdMaxC) {
        float* chan_ws = workspace + 4 * (size_t)kGnBwdMaxBatch * 32;
        const int C8 = C / 8;
        const int VC = C8 < 64 ? C8 : 64;                 // 8-channel vectors per block (512 channels)
        const int chunks = ceil_div(C8, VC);
        const int R = 256 / VC;
        const int threads = ceil_div(R * VC, 32) * 32;
        int slabs = ceil_div(kGnBwdMaxSlabs - 48, batch * chunks);   // ~4 CTAs per SM on 148 SMs, bounded by the scratch size
        int pps = ceil_div(hw, slabs);
        if (pps < 2 * R) pps = 2 * R;
        slabs = ceil_div(hw, pps);
        const size_t smem = (size_t)2 * R * VC * 8 * sizeof(float);
        if (in_dtype == B200SD_F32)
            gn_bwd_partial_kernel<B200SD_F32><<<dim3(slabs, chunks, batch), dim3(threads), smem, s>>>(x0, x1, C0, C1, gamma,
                                      beta, static_cast<const bf16*>(dy), mean_rstd, chan_ws, hw, groups, silu, VC, pps);
        else
            gn_bwd_partial_kernel<B200SD_BF16><<<dim3(slabs, chunks, batch), dim3(threads), smem, s>>>(x0, x1, C0, C1, gamma,
                                      beta, static_cast<const bf16*>(dy), mean_rstd, chan_ws, hw, groups, silu, VC, pps);
        COUNT_LAUNCH();
        B200SD_LAUNCH_CHECK();
        {
            const int nE = 2 * cpg;
            const int parts = 256 / nE > 0 ? 256 / nE : 1;
            gn_bwd_finalize_kernel<<<dim3(groups, batch), dim3(256), (size_t)(parts + 1) * nE * sizeof(float), s>>>(gamma,
                                      mean_rstd, chan_ws, stats, dgamma, dbeta, C, hw, groups, slabs);
        }
        COUNT_LAUNCH();
        B200SD_LAUNCH_CHECK();
    } else {
        int threads = (512 / cpg) * cpg;
        if (threads / cpg > hw) threads = hw * cpg;
        threads = ceil_div(threads, 32) * 32;
        if (threads < 128) threads = 128;
        const size_t smem = (size_t)4 * threads * sizeof(float);
        if (in_dtype == B200SD_F32)
            gn_bwd_stats_kernel<B200SD_F32><<<dim3(groups, batch), dim3(threads), smem, s>>>(x0, x1, C0, C1, gamma, beta,
                                      static_cast<const bf16*>(dy), dgamma, dbeta, stats, hw, groups, eps, silu);
        else
            gn_bwd_stats_kernel<B200SD_BF16><<<dim3(groups, batch), dim3(threads), smem, s>>>(x0, x1, C0, C1, gamma, beta,
                                      static_cast<const bf16*>(dy), dgamma, dbeta, stats, hw, groups, eps, silu);
        COUNT_LAUNCH();
        B200SD_LAUNCH_CHECK();
    }
    {
        int blocks = ceil_div(b200sd_num_sms() * 4, batch);
        int ppb = ceil_div(hw, blocks);
        const int min_ppb = ceil_div(256 * 2, C / 8);
        if (ppb < min_ppb) ppb = min_ppb;
        blocks = ceil_div(hw, ppb);
        const dim3 grid(blocks, batch);
#define GN_BWD_APPLY(DT, ODT)                                                                                                   \
    gn_bwd_apply_kernel<DT, ODT><<<grid, dim3(256), 0, s>>>(x0, x1, C0, C1, gamma, beta,                    \
                              static_cast<const bf16*>(dy), add_src, out0, out1, accumulate0, accumulate1,                       \
                              static_cast<const float4*>(stats), hw, groups, silu, ppb)
        if (in_dtype == B200SD_F32 && out_dtype == B200SD_F32) GN_BWD_APPLY(B200SD_F32, B200SD_F32);
        else if (in_dtype == B200SD_F32) GN_BWD_APPLY(B200SD_F32, B200SD_BF16);
        else if (out_dtype == B200SD_F32) GN_BWD_APPLY(B200SD_BF16, B200SD_F32);
        else GN_BWD_APPLY(B200SD_BF16, B200SD_BF16);
#undef GN_BWD_APPLY
        COUNT_LAUNCH();
        B200SD_LAUNCH_CHECK();
    }
    return B200SD_OK;
}

extern "C" int b200sd_layernorm_bwd(const void* x, int in_dtype, const float* gamma, const void* dy, float* dres,
                                    float* dgamma, float* dbeta, int rows, int C, float eps, b200sd_stream_t stream) {
    B200SD_REQUIRE(x && gamma && dy && dres, "layernorm_bwd: null pointer");
    B200SD_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), "layernorm_bwd: dgamma / dbeta must both be given or both NULL");
    B200SD_REQUIRE(rows > 0 && C % 64 == 0 && C >= 64 && C <= 1280, "layernorm_bwd: C=%d unsupported (multiple of 64, <= 1280)", C);
    B200SD_REQUIRE(in_dtype == B200SD_BF16 || in_dtype == B200SD_F32, "layernorm_bwd: bad input dtype");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int blocks = b200sd_num_sms() * 2;
    int rpb = ceil_div(rows, blocks);
    if (rpb < 8) rpb = 8;
    blocks = ceil_div(rows, rpb);
    const size_t smem = (size_t)8 * C * sizeof(float);
    const bf16* dyb = static_cast<const bf16*>(dy);
#define LNB_CASE(P)                                                                                                              \
    case P:                                                                                                                      \
        if (in_dtype == B200SD_F32)                                                                                              \
            layernorm_bwd_kernel<P, B200SD_F32><<<dim3(blocks), dim3(256), smem, s>>>(x, gamma, dyb, dres, dgamma, dbeta, rows, C, eps, rpb); \
        else                                                                                                                     \
            layernorm_bwd_kernel<P, B200SD_BF16><<<dim3(blocks), dim3(256), smem, s>>>(x, gamma, dyb, dres, dgamma, dbeta, rows, C, eps, rpb); \
        break;
    switch (C / 64) {
        LNB_CASE(1) LNB_CASE(2) LNB_CASE(3) LNB_CASE(4) LNB_CASE(5) LNB_CASE(6) LNB_CASE(7) LNB_CASE(8) LNB_CASE(9) LNB_CASE(10)
        LNB_CASE(11) LNB_CASE(12) LNB_CASE(13) LNB_CASE(14) LNB_CASE(15) LNB_CASE(16) LNB_CASE(17) LNB_CASE(18) LNB_CASE(19) LNB_CASE(20)
        default:
            B200SD_REQUIRE(false, "layernorm_bwd: C=%d unsupported", C);
    }
#undef LNB_CASE
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_geglu_fwd(const void* u, void* out, int64_t rows, int C_half, b200sd_stream_t stream) {
    B200SD_REQUIRE(u && out && rows > 0 && C_half > 0 && C_half % 8 == 0, "geglu_fwd: bad arguments");
    geglu_fwd_kernel<<<dim3(ew_grid(rows * (C_half / 8), 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(u), static_cast<bf16*>(out), rows, C_half / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_geglu_bwd(const void* u, const void* dff, void* du, int64_t rows, int C_half, b200sd_stream_t stream) {
    B200SD_REQUIRE(u && dff && du && rows > 0 && C_half > 0 && C_half % 8 == 0, "geglu_bwd: bad arguments");
    geglu_bwd_kernel<<<dim3(ew_grid(rows * (C_half / 8), 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(u), static_cast<const bf16*>(dff), static_cast<bf16*>(du), rows, C_half / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_upsample2x_bwd(const void* dy, float* dx, int batch, int H, int W, int C, int accumulate,
                                     b200sd_stream_t stream) {
    B200SD_REQUIRE(dy && dx && C % 8 == 0 && batch > 0 && H > 0 && W > 0, "upsample2x_bwd: bad arguments");
    const int64_t total = (int64_t)batch * H * W * (C / 8);
    upsample2x_bwd_kernel<<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(dy), dx, batch, H, W, C / 8, accumulate);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_col2im_s2(const void* dcol, float* dx, int batch, int H, int W, int C, int accumulate,
                                b200sd_stream_t stream) {
    B200SD_REQUIRE(dcol && dx && C % 8 == 0 && batch > 0 && H % 2 == 0 && W % 2 == 0, "col2im_s2: bad arguments");
    const int64_t total = (int64_t)batch * H * W * (C / 8);
    col2im_s2_kernel<<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(dcol), dx, batch, H, W, C / 8, accumulate);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_conv_out_bwd(const float* dout_nchw, const void* x_nhwc, const float* w, void* dx_nhwc, float* dw,
                                   float* dbias, int batch, int Cin, int Cout, int H, int W, b200sd_stream_t stream) {
    B200SD_REQUIRE(dout_nchw && w && dx_nhwc, "conv_out_bwd: null pointer");
    B200SD_REQUIRE(Cout >= 1 && Cout <= 4 && Cin % 8 == 0 && batch > 0 && H > 0 && W > 0, "conv_out_bwd: bad sizes");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t total = (int64_t)batch * H * W * (Cin / 8);
    conv_out_dgrad_kernel<<<dim3(ew_grid(total, 256)), dim3(256), 0, s>>>(dout_nchw, w,
                              static_cast<bf16*>(dx_nhwc), batch, Cin, Cout, H, W);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    if (dw != nullptr) {
        B200SD_REQUIRE(x_nhwc != nullptr && dbias != nullptr, "conv_out_bwd: x / dbias missing");
        const int pix = batch * H * W;
        int ppb = ceil_div(pix, b200sd_num_sms() * 2);
        if (ppb < 16) ppb = 16;
        conv_small_wgrad_kernel<B200SD_BF16><<<dim3(ceil_div(pix, ppb), ceil_div(Cin, 256)), dim3(256), 0, s>>>(x_nhwc,
                                  dout_nchw, dw, batch, H, W, Cin, Cout, -1, 1, ppb);
        COUNT_LAUNCH();
        B200SD_LAUNCH_CHECK();
        nchw_channel_sum_kernel<<<dim3(Cout), dim3(256), 0, s>>>(dout_nchw, dbias, batch, Cout, H * W);
        COUNT_LAUNCH();
    }
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_conv_in_wgrad(const void* dy_nhwc, int dy_dtype, const float* x_nchw, float* dw, int batch, int Cin,
                                    int Cout, int H, int W, b200sd_stream_t stream) {
    B200SD_REQUIRE(dy_nhwc && x_nchw && dw, "conv_in_wgrad: null pointer");
    B200SD_REQUIRE(Cin >= 1 && Cin <= 4 && batch > 0 && H > 0 && W > 0, "conv_in_wgrad: bad sizes");
    B200SD_REQUIRE(dy_dtype == B200SD_BF16 || dy_dtype == B200SD_F32, "conv_in_wgrad: bad dtype");
    const int pix = batch * H * W;
    int ppb = ceil_div(pix, b200sd_num_sms() * 2);
    if (ppb < 16) ppb = 16;
    const dim3 grid(ceil_div(pix, ppb), ceil_div(Cout, 256));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (dy_dtype == B200SD_F32)
        conv_small_wgrad_kernel<B200SD_F32><<<grid, dim3(256), 0, s>>>(dy_nhwc, x_nchw, dw, batch, H, W, Cout, Cin, 1, 0, ppb);
    else
        conv_small_wgrad_kernel<B200SD_BF16><<<grid, dim3(256), 0, s>>>(dy_nhwc, x_nchw, dw, batch, H, W, Cout, Cin, 1, 0, ppb);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_cast_act(const float* in, void* out_bf16, int64_t n, int silu, b200sd_stream_t stream) {
    B200SD_REQUIRE(in && out_bf16 && n > 0, "cast_act: bad arguments");
    cast_act_kernel<<<dim3(ew_grid(n, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(in,
                              static_cast<bf16*>(out_bf16), n, silu);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_silu_bwd_mul(const float* pre, float* grad, int64_t n, b200sd_stream_t stream) {
    B200SD_REQUIRE(pre && grad && n > 0, "silu_bwd_mul: bad arguments");
    silu_bwd_mul_kernel<<<dim3(ew_grid(n, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(pre, grad, n);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_cast_flat(const float* in, void* out_bf16, int64_t n, b200sd_stream_t stream) {
    B200SD_REQUIRE(in && out_bf16 && n > 0 && n % 8 == 0, "cast_flat: n must be a positive multiple of 8");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out_bf16)) & 15) == 0, "cast_flat: pointers must be 16-byte aligned");
    cast_flat_kernel<<<dim3(ew_grid(n / 8, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(in,
                              static_cast<bf16*>(out_bf16), n / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_adamw_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, void* weights_bf16, int64_t n,
                                 float lr, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                                 int zero_grad, b200sd_stream_t stream) {
    B200SD_REQUIRE(param && grad && exp_avg && exp_avg_sq && weights_bf16, "adamw_step: null pointer");
    B200SD_REQUIRE(n > 0 && n % 4 == 0 && step >= 1, "adamw_step: n must be a positive multiple of 4 and step >= 1");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(exp_avg) |
                     reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0 && (reinterpret_cast<uintptr_t>(weights_bf16) & 7) == 0,
                   "adamw_step: pointers must be 16-byte aligned");
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    adamw_flat_kernel<<<dim3(ew_grid(n / 4, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(param, grad,
                              exp_avg, exp_avg_sq, static_cast<bf16*>(weights_bf16), n / 4, lr, beta1, beta2, eps, weight_decay,
                              (float)bc1, (float)(1.0 / sqrt(bc2)), grad_scale, zero_grad);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
