// b200sd -- the small kernels around the GEMMs: timestep embedding, time-MLP linears, the two
// degenerate convs at the ends of the UNet (4 -> 320 and 320 -> 4 channels), nearest x2 upsample
// and the stride-2 im2col of the three Downsample2D convs.
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

// ---- sinusoidal timestep embedding (fp32, accurate sin/cos: arguments reach ~1000 rad) -----------
__global__ void temb_kernel(const float* __restrict__ t, float* __restrict__ out, int batch, int dim) {
    const int half = dim / 2;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch * half) return;
    const int b = i / half, j = i % half;
    const float expo = (-9.210340371976184f * (float)j) / (float)half;  // -ln(10000) * j / half
    const float arg = t[b] * expf(expo);
    out[(size_t)b * dim + j] = cosf(arg);         // flip_sin_to_cos = True: cos first
    out[(size_t)b * dim + half + j] = sinf(arg);
}

// ---- small-M linear: one warp per output feature, up to 8 batch rows at a time --------------------
// kSlRows = batch rows handled per CTA (template: CFG batch 2 must not pay for 8 rows of accumulators and staging)
template <int kSlRows>
__global__ void __launch_bounds__(256) small_linear_kernel(const float* __restrict__ in, const bf16* __restrict__ w,
                                                           const float* __restrict__ bias, float* __restrict__ out,
                                                           int batch, int N, int K, int silu_in, int silu_out) {
    extern __shared__ float s_in[];  // [kSlRows][K]
    const int b0 = blockIdx.y * kSlRows;
    const int nb = min(kSlRows, batch - b0);
    for (int i = threadIdx.x; i < kSlRows * K; i += blockDim.x) {
        const int r = i / K, k = i % K;
        float v = 0.f;
        if (r < nb) {
            v = in[(size_t)(b0 + r) * K + k];
            if (silu_in) v = v / (1.0f + expf(-v));
        }
        s_in[i] = v;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warps_total = gridDim.x * 8;
    constexpr int NF = 4;  // output features per warp pass: NF independent 16-byte weight loads in flight per lane
    for (int n0 = (blockIdx.x * 8 + warp) * NF; n0 < N; n0 += warps_total * NF) {
        float acc[NF][kSlRows];
#pragma unroll
        for (int f = 0; f < NF; ++f)
#pragma unroll
            for (int r = 0; r < kSlRows; ++r) acc[f][r] = 0.f;
#pragma unroll 5
        for (int v8 = lane; v8 < K / 8; v8 += 32) {   // K = 1280: 5 x NF 16-byte weight loads in flight per lane
            uint4 u[NF];
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                const int n = min(n0 + f, N - 1);
                u[f] = __ldg(reinterpret_cast<const uint4*>(w + (size_t)n * K) + v8);
            }
            float xr[kSlRows][8];
#pragma unroll
            for (int r = 0; r < kSlRows; ++r) {
                const float4 x0 = *reinterpret_cast<const float4*>(s_in + r * K + v8 * 8);
                const float4 x1 = *reinterpret_cast<const float4*>(s_in + r * K + v8 * 8 + 4);
                xr[r][0] = x0.x; xr[r][1] = x0.y; xr[r][2] = x0.z; xr[r][3] = x0.w;
                xr[r][4] = x1.x; xr[r][5] = x1.y; xr[r][6] = x1.z; xr[r][7] = x1.w;
            }
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                float wf[8];
                float2 t;
                t = unpack_bf16x2(u[f].x); wf[0] = t.x; wf[1] = t.y;
                t = unpack_bf16x2(u[f].y); wf[2] = t.x; wf[3] = t.y;
                t = unpack_bf16x2(u[f].z); wf[4] = t.x; wf[5] = t.y;
                t = unpack_bf16x2(u[f].w); wf[6] = t.x; wf[7] = t.y;
#pragma unroll
                for (int r = 0; r < kSlRows; ++r)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[f][r] += wf[j] * xr[r][j];
            }
        }
#pragma unroll
        for (int f = 0; f < NF; ++f)
#pragma unroll
            for (int r = 0; r < kSlRows; ++r) acc[f][r] = warp_sum(acc[f][r]);
        if (lane == 0) {
            for (int f = 0; f < NF && n0 + f < N; ++f) {
                const float bv = bias ? bias[n0 + f] : 0.f;
                for (int r = 0; r < nb; ++r) {
                    float v = acc[f][r] + bv;
                    if (silu_out) v = v / (1.0f + expf(-v));
                    out[(size_t)(b0 + r) * N + n0 + f] = v;
                }
            }
        }
    }
}

// ---- conv_in: NCHW fp32 (Cin = 4) -> NHWC bf16; thread = output-channel pair, block = 32 pixels ---
constexpr int kCinPix = 32;
template <int ODT>
__global__ void conv_in_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                               void* __restrict__ out, int batch, int Cout, int H, int W) {
    constexpr int Cin = 4;
    __shared__ float patch[kCinPix][9 * Cin];
    const int hw = H * W;
    const int pix0 = blockIdx.x * kCinPix;
    const int total = batch * hw;
    for (int i = threadIdx.x; i < kCinPix * 9 * Cin; i += blockDim.x) {
        const int pl = i / (9 * Cin), r = i % (9 * Cin);
        const int tap = r / Cin, c = r % Cin;
        const int pix = pix0 + pl;
        float v = 0.f;
        if (pix < total) {
            const int b = pix / hw, rem = pix % hw;
            const int y = rem / W + tap / 3 - 1, xx = rem % W + tap % 3 - 1;
            if (y >= 0 && y < H && xx >= 0 && xx < W) v = x[((size_t)(b * Cin + c) * H + y) * W + xx];
        }
        patch[pl][r] = v;
    }
    __syncthreads();
    for (int co2 = threadIdx.x; co2 < Cout / 2; co2 += blockDim.x) {
        const int co = co2 * 2;
        float w0[9 * Cin], w1[9 * Cin];
#pragma unroll
        for (int r = 0; r < 9 * Cin; ++r) {  // packed [Cout][tap][Cin]
            w0[r] = __ldg(w + (size_t)co * 9 * Cin + r);
            w1[r] = __ldg(w + (size_t)(co + 1) * 9 * Cin + r);
        }
        const float b0 = bias[co], b1 = bias[co + 1];
        for (int pl = 0; pl < kCinPix; ++pl) {
            const int pix = pix0 + pl;
            if (pix >= total) break;
            float a0 = b0, a1 = b1;
#pragma unroll
            for (int r = 0; r < 9 * Cin; ++r) {
                const float v = patch[pl][r];
                a0 += w0[r] * v;
                a1 += w1[r] * v;
            }
            if constexpr (ODT == B200SD_F32)
                *reinterpret_cast<float2*>(static_cast<float*>(out) + (size_t)pix * Cout + co) = make_float2(a0, a1);
            else
                *reinterpret_cast<uint32_t*>(static_cast<bf16*>(out) + (size_t)pix * Cout + co) = pack_bf16x2(a0, a1);
        }
    }
}

// ---- conv_out: NHWC bf16 (Cin = 320) -> NCHW fp32 (Cout = 4); warp per pixel, lanes over channels -
constexpr int kCoutMax = 4;
constexpr int kCoCP = 5;   // channel pairs per lane of the unrolled path: Cin = 64 * kCoCP = 320
__global__ void __launch_bounds__(256) conv_out_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                                       const float* __restrict__ bias, float* __restrict__ out,
                                                       int batch, int Cin, int Cout, int H, int W, int pix_per_warp) {
    extern __shared__ float s_w[];  // packed [Cout][tap][Cin]
    for (int i = threadIdx.x; i < Cout * 9 * Cin / 4; i += blockDim.x)   // static weights: before the wait (Cin % 4 == 0)
        reinterpret_cast<float4*>(s_w)[i] = __ldg(reinterpret_cast<const float4*>(w) + i);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int hw = H * W, total = batch * hw;
    const int first = (blockIdx.x * 8 + warp) * pix_per_warp;
    for (int pix = first; pix < min(first + pix_per_warp, total); ++pix) {
        const int b = pix / hw, rem = pix % hw, y = rem / W, xx = rem % W;
        float acc[kCoutMax] = {0.f, 0.f, 0.f, 0.f};
        if (Cin == 64 * kCoCP) {
            // SD's conv_out (Cin = 320): issue the loads of all 9 taps before any arithmetic -- one memory latency per pixel
            // instead of one per tap (the kernel was latency-bound: 45 us for 94 MFLOP)
            uint32_t v[9][kCoCP];
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                const int yy = y + tap / 3 - 1, xs = xx + tap % 3 - 1;
                const bool ok = yy >= 0 && yy < H && xs >= 0 && xs < W;
                const uint32_t* src = reinterpret_cast<const uint32_t*>(x + ((size_t)(b * H + (ok ? yy : y)) * W + (ok ? xs : xx)) * Cin);
#pragma unroll
                for (int i = 0; i < kCoCP; ++i) v[tap][i] = ok ? __ldg(src + lane + 32 * i) : 0u;
            }
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
                for (int i = 0; i < kCoCP; ++i) {
                    const float2 f = unpack_bf16x2(v[tap][i]);
#pragma unroll
                    for (int co = 0; co < kCoutMax; ++co) {
                        if (co < Cout) {
                            const float2 wv = *reinterpret_cast<const float2*>(s_w + (size_t)(co * 9 + tap) * Cin + 2 * (lane + 32 * i));
                            acc[co] += f.x * wv.x + f.y * wv.y;
                        }
                    }
                }
            }
        } else {
            for (int tap = 0; tap < 9; ++tap) {
                const int yy = y + tap / 3 - 1, xs = xx + tap % 3 - 1;
                if (yy < 0 || yy >= H || xs < 0 || xs >= W) continue;
                const uint32_t* src = reinterpret_cast<const uint32_t*>(x + ((size_t)(b * H + yy) * W + xs) * Cin);
                for (int c2 = lane; c2 < Cin / 2; c2 += 32) {
                    const float2 f = unpack_bf16x2(__ldg(src + c2));
#pragma unroll
                    for (int co = 0; co < kCoutMax; ++co) {
                        if (co < Cout) {
                            const float* wp = s_w + (size_t)(co * 9 + tap) * Cin + 2 * c2;
                            acc[co] += f.x * wp[0] + f.y * wp[1];
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int co = 0; co < kCoutMax; ++co) acc[co] = warp_sum(acc[co]);
        if (lane == 0)
            for (int co = 0; co < Cout; ++co) out[((size_t)(b * Cout + co) * H + y) * W + xx] = acc[co] + bias[co];
    }
}

// ---- nearest x2 upsample, NHWC, 8-channel vectors (fp32 or bf16 in, bf16 out) -----------------------
template <int DT>
__global__ void upsample2x_kernel(const void* __restrict__ x, bf16* __restrict__ out, int batch, int H, int W, int C8) {
    const int64_t total = (int64_t)batch * 4 * H * W * C8;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i % C8);
        int64_t p = i / C8;
        const int ox = (int)(p % (2 * W));
        p /= (2 * W);
        const int oy = (int)(p % (2 * H));
        const int b = (int)(p / (2 * H));
        float v[8];
        ld8<DT>(x, (size_t)(((int64_t)(b * H + (oy >> 1)) * W + (ox >> 1)) * C8 + c) * 8, v);
        st8<B200SD_BF16>(out, (size_t)i * 8, v);
    }
}

// ---- im2col for the stride-2 pad-1 3x3 Downsample2D conv --------------------------------------------
template <int DT>
__global__ void im2col_s2_kernel(const void* __restrict__ x, bf16* __restrict__ out, int batch, int H, int W, int C8, int pad) {
    const int OH = H / 2, OW = W / 2;
    const int64_t total = (int64_t)batch * OH * OW * 9 * C8;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i % C8);
        int64_t p = i / C8;
        const int tap = (int)(p % 9);
        p /= 9;
        const int ox = (int)(p % OW);
        p /= OW;
        const int oy = (int)(p % OH);
        const int b = (int)(p / OH);
        const int y = 2 * oy + tap / 3 - pad, xx = 2 * ox + tap % 3 - pad;   // pad 1: UNet Downsample2D; pad 0: the VAE's (0,1,0,1) padding
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (y >= 0 && y < H && xx >= 0 && xx < W) ld8<DT>(x, (size_t)(((int64_t)(b * H + y) * W + xx) * C8 + c) * 8, v);
        st8<B200SD_BF16>(out, (size_t)i * 8, v);
    }
}

int ew_grid(int64_t total, int threads) {
    int64_t blocks = (total + threads - 1) / threads;
    const int64_t cap = (int64_t)b200sd_num_sms() * 8;
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace

extern "C" int b200sd_timestep_embedding(const float* timesteps, float* out, int batch, int dim,
                                         b200sd_stream_t stream) {
    B200SD_REQUIRE(timesteps && out, "timestep_embedding: null pointer");
    B200SD_REQUIRE(batch > 0 && dim > 0 && dim % 2 == 0, "timestep_embedding: bad sizes");
    const int total = batch * dim / 2;
    temb_kernel<<<dim3(ceil_div(total, 128)), dim3(128), 0, static_cast<cudaStream_t>(stream)>>>(timesteps, out, batch, dim);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_small_linear(const float* in, const void* w_bf16, const float* bias, float* out, int batch, int N,
                                   int K, int silu_in, int silu_out, b200sd_stream_t stream) {
    B200SD_REQUIRE(in && w_bf16 && out, "small_linear: null pointer");
    B200SD_REQUIRE(batch > 0 && N > 0 && K > 0 && K % 8 == 0, "small_linear: bad sizes (K must be a multiple of 8)");
    const int rows = batch <= 2 ? 2 : (batch <= 4 ? 4 : 8);
    const size_t smem = (size_t)rows * K * sizeof(float);
    B200SD_REQUIRE(smem <= 96 * 1024, "small_linear: K=%d too large", K);
    B200SD_CUDA(b200sd_opt_in_smem(small_linear_kernel<2>, 96 * 1024));
    B200SD_CUDA(b200sd_opt_in_smem(small_linear_kernel<4>, 96 * 1024));
    B200SD_CUDA(b200sd_opt_in_smem(small_linear_kernel<8>, 96 * 1024));
    int gx = ceil_div(N, 8 * 4);
    const int cap = b200sd_num_sms() * 4;
    if (gx > cap) gx = cap;
    dim3 grid(gx, ceil_div(batch, rows));
    auto kern = rows == 2 ? small_linear_kernel<2> : (rows == 4 ? small_linear_kernel<4> : small_linear_kernel<8>);
    kern<<<dim3(grid), dim3(256), smem, static_cast<cudaStream_t>(stream)>>>(in, static_cast<const bf16*>(w_bf16), bias,
                              out, batch, N, K, silu_in, silu_out);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_conv_in(const float* x_nchw, const float* w, const float* bias, void* out_nhwc, int batch, int Cin,
                              int Cout, int H, int W, int out_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(x_nchw && w && bias && out_nhwc, "conv_in: null pointer");
    B200SD_REQUIRE(Cin == 4, "conv_in: only Cin == 4 (SD latent) is supported, got %d", Cin);
    B200SD_REQUIRE(Cout % 2 == 0 && batch > 0 && H > 0 && W > 0, "conv_in: bad sizes");
    const int total = batch * H * W;
    int threads = Cout / 2;
    if (threads > 256) threads = 256;
    threads = ceil_div(threads, 32) * 32;
    if (out_dtype == B200SD_F32)
        conv_in_kernel<B200SD_F32><<<dim3(ceil_div(total, kCinPix)), dim3(threads), 0, static_cast<cudaStream_t>(stream)>>>(x_nchw, w, bias, out_nhwc, batch, Cout, H, W);
    else
        conv_in_kernel<B200SD_BF16><<<dim3(ceil_div(total, kCinPix)), dim3(threads), 0, static_cast<cudaStream_t>(stream)>>>(x_nchw, w, bias, out_nhwc, batch, Cout, H, W);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_conv_out(const void* x_nhwc, const float* w, const float* bias, float* out_nchw, int batch, int Cin,
                               int Cout, int H, int W, b200sd_stream_t stream) {
    B200SD_REQUIRE(x_nhwc && w && bias && out_nchw, "conv_out: null pointer");
    B200SD_REQUIRE(Cout >= 1 && Cout <= kCoutMax && Cin % 4 == 0, "conv_out: Cout must be <= 4 and Cin a multiple of 4");
    const size_t smem = (size_t)Cout * 9 * Cin * sizeof(float);
    B200SD_REQUIRE(smem <= 96 * 1024, "conv_out: Cin=%d too large", Cin);
    B200SD_CUDA(b200sd_opt_in_smem(conv_out_kernel, 96 * 1024));
    const int total = batch * H * W;
    int ppw = ceil_div(total, b200sd_num_sms() * 2 * 8);
    if (ppw < 4) ppw = 4;
    const int blocks = ceil_div(total, ppw * 8);
    conv_out_kernel<<<dim3(blocks), dim3(256), smem, static_cast<cudaStream_t>(stream)>>>(static_cast<const bf16*>(x_nhwc), w, bias,
                                                                             out_nchw, batch, Cin, Cout, H, W, ppw);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// [M][ld] fp32 (NHWC, the first C of ld columns) + bias -> NCHW fp32: the tail of the tensor-core conv_out
__global__ void __launch_bounds__(256) nhwc_bias_to_nchw_kernel(const float* __restrict__ x, const float* __restrict__ bias,
                                                                float* __restrict__ out, int total, int hw, int C, int ld) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= total) return;
    const int b = m / hw, pix = m - b * hw;
    const float4 v = __ldg(reinterpret_cast<const float4*>(x + (size_t)m * ld));
    const float4 u = C > 4 ? __ldg(reinterpret_cast<const float4*>(x + (size_t)m * ld) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float vv[8] = {v.x, v.y, v.z, v.w, u.x, u.y, u.z, u.w};
    for (int c = 0; c < C; ++c) out[((size_t)b * C + c) * hw + pix] = vv[c] + __ldg(bias + c);
}

extern "C" int b200sd_nhwc_bias_to_nchw(const float* x, const float* bias, float* out_nchw, int batch, int C, int hw, int ld,
                                        b200sd_stream_t stream) {
    B200SD_REQUIRE(x && bias && out_nchw, "nhwc_bias_to_nchw: null pointer");
    B200SD_REQUIRE(C >= 1 && C <= 8 && ld % 4 == 0 && ld >= (C > 4 ? 8 : 4) && batch > 0 && hw > 0, "nhwc_bias_to_nchw: C in 1..8, ld %% 4 == 0");
    const int total = batch * hw;
    nhwc_bias_to_nchw_kernel<<<dim3(ceil_div(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x, bias,
                              out_nchw, total, hw, C, ld);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_upsample2x(const void* x, void* out, int batch, int H, int W, int C, int in_dtype,
                                 b200sd_stream_t stream) {
    B200SD_REQUIRE(x && out, "upsample2x: null pointer");
    B200SD_REQUIRE(C % 8 == 0 && batch > 0 && H > 0 && W > 0, "upsample2x: bad sizes");
    const int64_t total = (int64_t)batch * 4 * H * W * (C / 8);
    if (in_dtype == B200SD_F32)
        upsample2x_kernel<B200SD_F32><<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<bf16*>(out), batch, H, W, C / 8);
    else
        upsample2x_kernel<B200SD_BF16><<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<bf16*>(out), batch, H, W, C / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_im2col_s2(const void* x, void* out, int batch, int H, int W, int C, int in_dtype,
                                b200sd_stream_t stream) {
    return b200sd_im2col_s2_pad(x, out, batch, H, W, C, in_dtype, 1, stream);
}

extern "C" int b200sd_im2col_s2_pad(const void* x, void* out, int batch, int H, int W, int C, int in_dtype, int pad,
                                    b200sd_stream_t stream) {
    B200SD_REQUIRE(x && out, "im2col_s2: null pointer");
    B200SD_REQUIRE(pad == 0 || pad == 1, "im2col_s2: pad must be 0 (pad right/bottom only) or 1 (symmetric)");
    B200SD_REQUIRE(C % 8 == 0 && batch > 0 && H % 2 == 0 && W % 2 == 0, "im2col_s2: bad sizes");
    const int64_t total = (int64_t)batch * (H / 2) * (W / 2) * 9 * (C / 8);
    if (in_dtype == B200SD_F32)
        im2col_s2_kernel<B200SD_F32><<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<bf16*>(out), batch, H, W, C / 8, pad);
    else
        im2col_s2_kernel<B200SD_BF16><<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<bf16*>(out), batch, H, W, C / 8, pad);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
