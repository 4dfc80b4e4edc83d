// b200sd -- the kernels of AutoencoderKL (SURVEY.md 8f N1; reference call sites finetune_sd.py:325-327, 460-462 and the decode
// inside every `pipeline(...)` call, inference.py:175-176) that the UNet does not already have: the row softmax of the
// single-head 512-channel attention of the mid block (its two contractions run as tcgen05 GEMMs over a materialised score
// matrix: S x S fp32 never leaves L2 at S = 4096), the 1x1 quant / post-quant convolutions over the 4 / 8 latent channels, and
// the posterior sample mean + exp(0.5 logvar) * noise.  Everything else of the VAE is the UNet's kernels at C = 128 / 256 / 512:
// implicit-GEMM conv3x3 (image rows wider than a tile: gemm_tcgen05.cu `tiles_x`), GroupNorm+SiLU, nearest upsample, the
// stride-2 im2col (pad 0), the 4-channel end convs.
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

__device__ __forceinline__ float block_reduce(float v, float* sh, bool is_max) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float t = __shfl_xor_sync(0xffffffffu, v, o);
        v = is_max ? fmaxf(v, t) : v + t;
    }
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    float r = sh[0];
    for (int i = 1; i < nw; ++i) r = is_max ? fmaxf(r, sh[i]) : r + sh[i];
    return r;
}

// out[r][:] = softmax(scale * x[r][:])  (fp32 -> bf16); one CTA per row, the row is read three times (L2-resident)
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ x, bf16* __restrict__ out, int L, int ldx,
                                                           int ldo, float scale_log2) {
    __shared__ float sh[8];
    const float4* xr = reinterpret_cast<const float4*>(x + (size_t)blockIdx.x * ldx);
    const int L4 = L >> 2;
    float m = -INFINITY;
    for (int i = threadIdx.x; i < L4; i += blockDim.x) {
        const float4 v = xr[i];
        m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
    }
    m = block_reduce(m, sh, true) * scale_log2;
    float s = 0.f;
    for (int i = threadIdx.x; i < L4; i += blockDim.x) {
        const float4 v = xr[i];
        s += exp2f(v.x * scale_log2 - m) + exp2f(v.y * scale_log2 - m) + exp2f(v.z * scale_log2 - m) + exp2f(v.w * scale_log2 - m);
    }
    const float inv = 1.f / block_reduce(s, sh, false);
    uint2* orow = reinterpret_cast<uint2*>(out + (size_t)blockIdx.x * ldo);
    for (int i = threadIdx.x; i < L4; i += blockDim.x) {
        const float4 v = xr[i];
        orow[i] = make_uint2(pack_bf16x2(exp2f(v.x * scale_log2 - m) * inv, exp2f(v.y * scale_log2 - m) * inv),
                             pack_bf16x2(exp2f(v.z * scale_log2 - m) * inv, exp2f(v.w * scale_log2 - m) * inv));
    }
}

// 1x1 convolution over a handful of channels, NCHW fp32 -> NCHW fp32 (quant_conv 8 -> 8, post_quant_conv 4 -> 4)
__global__ void conv1x1_small_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                     float* __restrict__ out, int batch, int Cin, int Cout, int hw) {
    const int64_t total = (int64_t)batch * hw, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int b = (int)(i / hw), p = (int)(i % hw);
        float v[8];
        for (int c = 0; c < Cin; ++c) v[c] = x[((size_t)b * Cin + c) * hw + p];
        for (int o = 0; o < Cout; ++o) {
            float acc = bias[o];
            for (int c = 0; c < Cin; ++c) acc = fmaf(w[o * Cin + c], v[c], acc);
            out[((size_t)b * Cout + o) * hw + p] = acc;
        }
    }
}

// DiagonalGaussianDistribution.sample(): moments NCHW [batch][2C][hw] = [mean | logvar]; out = (mean + exp(0.5 clamp(logvar,
// -30, 20)) * noise) * out_scale  (noise == NULL: the mode)
__global__ void gaussian_sample_kernel(const float* __restrict__ moments, const float* __restrict__ noise, float* __restrict__ out,
                                       int batch, int C, int hw, float out_scale) {
    const int64_t total = (int64_t)batch * C * hw, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t b = i / ((int64_t)C * hw), r = i % ((int64_t)C * hw);
        const float mean = moments[b * 2 * C * hw + r];
        float v = mean;
        if (noise != nullptr) {
            const float lv = fminf(fmaxf(moments[b * 2 * C * hw + (int64_t)C * hw + r], -30.f), 20.f);
            v = fmaf(expf(0.5f * lv), noise[i], mean);
        }
        out[i] = v * out_scale;
    }
}

inline int ew_grid(int64_t n, int threads) {
    int64_t blocks = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)b200sd_num_sms() * 8;
    return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

}  // namespace

extern "C" int b200sd_softmax_rows(const float* x, void* out_bf16, int rows, int L, int ldx, int ldo, float scale,
                                   b200sd_stream_t stream) {
    B200SD_REQUIRE(x && out_bf16 && rows > 0 && L > 0, "softmax_rows: bad arguments");
    B200SD_REQUIRE(L % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0, "softmax_rows: L / ldx / ldo must be multiples of 4");
    softmax_rows_kernel<<<dim3(rows), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x,
                              static_cast<bf16*>(out_bf16), L, ldx, ldo, scale * 1.4426950408889634f);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_conv1x1_small(const float* x_nchw, const float* w, const float* bias, float* out_nchw, int batch, int Cin,
                                    int Cout, int hw, b200sd_stream_t stream) {
    B200SD_REQUIRE(x_nchw && w && bias && out_nchw, "conv1x1_small: null pointer");
    B200SD_REQUIRE(batch > 0 && hw > 0 && Cin >= 1 && Cin <= 8 && Cout >= 1 && Cout <= 8, "conv1x1_small: 1..8 channels");
    conv1x1_small_kernel<<<dim3(ew_grid((int64_t)batch * hw, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x_nchw, w, bias, out_nchw, batch, Cin, Cout, hw);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_gaussian_sample(const float* moments, const float* noise, float* out, int batch, int C, int hw, float out_scale,
                                      b200sd_stream_t stream) {
    B200SD_REQUIRE(moments && out && batch > 0 && C > 0 && hw > 0, "gaussian_sample: bad arguments");
    gaussian_sample_kernel<<<dim3(ew_grid((int64_t)batch * C * hw, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(moments, noise, out, batch, C, hw, out_scale);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
