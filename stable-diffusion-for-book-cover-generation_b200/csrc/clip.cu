// b200sd -- the kernels of the CLIP text encoder (SURVEY.md 8f N3; reference call sites finetune_sd.py:322-324, 375-379, 477:
// `encoder_hidden_states = text_encoder(batch["input_ids"])[0]`, transformers' CLIPTextModel) that are not GEMMs:
// token + position embedding (and its scatter-add backward), causal multi-head attention over the 77 tokens (forward and
// backward; head dim <= 64), quick-GELU (forward / backward) and the fp32-output final LayerNorm.  The twelve layers' linears
// run on the tcgen05 GEMM / dgrad / wgrad kernels of gemm_tcgen05.cu; LayerNorm 1/2 on norm.cu's kernels.
//
// Sizes: 77 tokens x 768 channels per prompt -- every kernel here moves a few hundred KB.  They are bound by launch latency,
// not by a pipe; the design goal is "one launch per op, everything of one (prompt, head) in shared memory, deterministic".
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

constexpr int kMaxS = 96;     // tokens per prompt the attention kernels hold in shared memory (CLIP: 77)
constexpr int kMaxD = 64;     // head dim (CLIP ViT-L/14 text: 64)

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- embeddings: x[b*S + s][:] = tok[ids[b][s]][:] + pos[s][:]  (fp32) ------------------------------------------------
__global__ void clip_embed_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tok, const float* __restrict__ pos,
                                  float* __restrict__ out, int rows, int S, int C4, int vocab) {
    const int64_t total = (int64_t)rows * C4, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int row = (int)(i / C4), c = (int)(i % C4);
        int64_t id = ids[row];
        id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
        const float4 a = __ldg(reinterpret_cast<const float4*>(tok) + id * C4 + c);
        const float4 p = __ldg(reinterpret_cast<const float4*>(pos) + (int64_t)(row % S) * C4 + c);
        reinterpret_cast<float4*>(out)[i] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
    }
}

// backward: dpos[s] += sum_b dx[b][s] (fixed order over b), dtok[ids[b][s]] += dx[b][s] (fp32 atomics: a token may repeat)
__global__ void clip_embed_bwd_kernel(const int64_t* __restrict__ ids, const float* __restrict__ dx, float* __restrict__ dtok,
                                      float* __restrict__ dpos, int batch, int S, int C, int vocab) {
    const int s = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float acc = 0.f;
        for (int b = 0; b < batch; ++b) {
            const float g = dx[((size_t)b * S + s) * C + c];
            acc += g;
            int64_t id = ids[b * S + s];
            id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
            atomicAdd(dtok + id * C + c, g);
        }
        dpos[(size_t)s * C + c] += acc;
    }
}

// ---- quick-GELU: g = u * sigmoid(1.702 u) ---------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + __expf(-x)); }

__global__ void quick_gelu_fwd_kernel(const bf16* __restrict__ u, bf16* __restrict__ out, int64_t n8) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
        uint4 raw = __ldg(reinterpret_cast<const uint4*>(u) + i);
        const bf16* h = reinterpret_cast<const bf16*>(&raw);
        uint4 o;
        bf16* oh = reinterpret_cast<bf16*>(&o);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float x = __bfloat162float(h[j]);
            oh[j] = __float2bfloat16_rn(x * sigmoid_f(1.702f * x));
        }
        reinterpret_cast<uint4*>(out)[i] = o;
    }
}

__global__ void quick_gelu_bwd_kernel(const bf16* __restrict__ u, const bf16* __restrict__ dg, bf16* __restrict__ du, int64_t n8) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
        uint4 ru = __ldg(reinterpret_cast<const uint4*>(u) + i), rg = __ldg(reinterpret_cast<const uint4*>(dg) + i);
        const bf16* hu = reinterpret_cast<const bf16*>(&ru);
        const bf16* hg = reinterpret_cast<const bf16*>(&rg);
        uint4 o;
        bf16* oh = reinterpret_cast<bf16*>(&o);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float x = __bfloat162float(hu[j]), g = __bfloat162float(hg[j]);
            const float sg = sigmoid_f(1.702f * x);
            oh[j] = __float2bfloat16_rn(g * (sg + 1.702f * x * sg * (1.f - sg)));
        }
        reinterpret_cast<uint4*>(du)[i] = o;
    }
}

// ---- final LayerNorm with an fp32 result (the text context handed to the UNet / returned to the caller) --------------
__global__ void __launch_bounds__(256) layernorm_f32out_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, float* __restrict__ out, int rows,
                                                               int C, float eps) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= rows) return;
    const float* xr = x + (size_t)warp * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += xr[c];
    const float mean = warp_sum_f(s) / (float)C;
    float ss = 0.f;
    for (int c = lane; c < C; c += 32) {
        const float d = xr[c] - mean;
        ss += d * d;
    }
    const float rstd = rsqrtf(warp_sum_f(ss) / (float)C + eps);
    for (int c = lane; c < C; c += 32) out[(size_t)warp * C + c] = (xr[c] - mean) * rstd * gamma[c] + beta[c];
}

// ---- causal attention over one prompt: one CTA per (prompt, head), everything in shared memory ------------------------
// qkv: bf16 [batch*S][ld] with q at column q_off + h*D, k at k_off + h*D, v at v_off + h*D.
__device__ __forceinline__ void load_head(const bf16* __restrict__ base, int ld, int S, int D, float* __restrict__ dst) {
    const int D8 = D >> 3;
    for (int i = threadIdx.x; i < S * D8; i += blockDim.x) {
        const int r = i / D8, c = (i % D8) * 8;
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(base + (size_t)r * ld + c));
        const bf16* h = reinterpret_cast<const bf16*>(&raw);
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[r * (kMaxD + 1) + c + j] = __bfloat162float(h[j]);
    }
}

// p[i][j] = softmax_j(scale * q_i . k_j) over j <= i, 0 above the diagonal
__device__ __forceinline__ void causal_probs(const float* __restrict__ q, const float* __restrict__ k, float* __restrict__ p, int S,
                                             int D, float scale) {
    const int P = kMaxS + 1;
    for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
        const int i = e / S, j = e % S;
        float acc = 0.f;
        if (j <= i) {
            const float* qi = q + i * (kMaxD + 1);
            const float* kj = k + j * (kMaxD + 1);
            for (int c = 0; c < D; ++c) acc = fmaf(qi[c], kj[c], acc);
        }
        p[i * P + j] = acc * scale;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int i = warp; i < S; i += nw) {
        float m = -INFINITY;
        for (int j = lane; j <= i; j += 32) m = fmaxf(m, p[i * P + j]);
        m = warp_max_f(m);
        float s = 0.f;
        for (int j = lane; j < S; j += 32) {
            const float e = j <= i ? __expf(p[i * P + j] - m) : 0.f;
            p[i * P + j] = e;
            s += e;
        }
        const float inv = 1.f / warp_sum_f(s);
        for (int j = lane; j <= i; j += 32) p[i * P + j] *= inv;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256) clip_attention_fwd_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int S, int D,
                                                                 int ld, int ldo, int q_off, int k_off, int v_off, float scale) {
    extern __shared__ float sm[];
    float* q = sm;
    float* k = q + kMaxS * (kMaxD + 1);
    float* v = k + kMaxS * (kMaxD + 1);
    float* p = v + kMaxS * (kMaxD + 1);
    const int b = blockIdx.y, h = blockIdx.x;
    const bf16* base = qkv + (size_t)b * S * ld + h * D;
    load_head(base + q_off, ld, S, D, q);
    load_head(base + k_off, ld, S, D, k);
    load_head(base + v_off, ld, S, D, v);
    __syncthreads();
    causal_probs(q, k, p, S, D, scale);
    const int P = kMaxS + 1;
    for (int e = threadIdx.x; e < S * D; e += blockDim.x) {
        const int i = e / D, c = e % D;
        float acc = 0.f;
        for (int j = 0; j <= i; ++j) acc = fmaf(p[i * P + j], v[j * (kMaxD + 1) + c], acc);
        out[((size_t)b * S + i) * ldo + h * D + c] = __float2bfloat16_rn(acc);
    }
}

// backward: recomputes P; dP = dO V^T; dS = P o (dP - rowsum(P o dP)) * scale; dV = P^T dO; dK = dS^T Q; dQ = dS K
__global__ void __launch_bounds__(256) clip_attention_bwd_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ dout,
                                                                 bf16* __restrict__ dqkv, int S, int D, int ld, int lddo, int ldd,
                                                                 int q_off, int k_off, int v_off, float scale) {
    extern __shared__ float sm[];
    float* q = sm;
    float* k = q + kMaxS * (kMaxD + 1);
    float* v = k + kMaxS * (kMaxD + 1);
    float* go = v + kMaxS * (kMaxD + 1);
    float* p = go + kMaxS * (kMaxD + 1);
    float* ds = p + kMaxS * (kMaxS + 1);
    const int b = blockIdx.y, h = blockIdx.x;
    const bf16* base = qkv + (size_t)b * S * ld + h * D;
    load_head(base + q_off, ld, S, D, q);
    load_head(base + k_off, ld, S, D, k);
    load_head(base + v_off, ld, S, D, v);
    load_head(dout + (size_t)b * S * lddo + h * D, lddo, S, D, go);
    __syncthreads();
    causal_probs(q, k, p, S, D, scale);
    const int P = kMaxS + 1, R = kMaxD + 1;
    for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
        const int i = e / S, j = e % S;
        float acc = 0.f;
        if (j <= i)
            for (int c = 0; c < D; ++c) acc = fmaf(go[i * R + c], v[j * R + c], acc);
        ds[i * P + j] = acc;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int i = warp; i < S; i += nw) {
        float d = 0.f;
        for (int j = lane; j <= i; j += 32) d = fmaf(p[i * P + j], ds[i * P + j], d);
        d = warp_sum_f(d);
        for (int j = lane; j < S; j += 32) ds[i * P + j] = j <= i ? p[i * P + j] * (ds[i * P + j] - d) * scale : 0.f;
    }
    __syncthreads();
    bf16* dbase = dqkv + (size_t)b * S * ldd + h * D;
    for (int e = threadIdx.x; e < S * D; e += blockDim.x) {
        const int r = e / D, c = e % D;
        float dq = 0.f, dk = 0.f, dv = 0.f;
        for (int j = 0; j <= r; ++j) dq = fmaf(ds[r * P + j], k[j * R + c], dq);
        for (int i = r; i < S; ++i) {
            dk = fmaf(ds[i * P + r], q[i * R + c], dk);
            dv = fmaf(p[i * P + r], go[i * R + c], dv);
        }
        bf16* row = dbase + (size_t)r * ldd + c;
        row[q_off] = __float2bfloat16_rn(dq);
        row[k_off] = __float2bfloat16_rn(dk);
        row[v_off] = __float2bfloat16_rn(dv);
    }
}

inline int ew_grid(int64_t n, int threads) {
    int64_t blocks = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)b200sd_num_sms() * 8;
    return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

}  // namespace

extern "C" int b200sd_clip_embed(const int64_t* ids, const float* tok, const float* pos, float* out, int batch, int S, int C,
                                 int vocab, b200sd_stream_t stream) {
    B200SD_REQUIRE(ids && tok && pos && out, "clip_embed: null pointer");
    B200SD_REQUIRE(batch > 0 && S > 0 && C > 0 && C % 4 == 0 && vocab > 0, "clip_embed: bad sizes");
    const int64_t total = (int64_t)batch * S * (C / 4);
    clip_embed_kernel<<<dim3(ew_grid(total, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(ids, tok,
                              pos, out, batch * S, S, C / 4, vocab);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_clip_embed_bwd(const int64_t* ids, const float* dx, float* dtok, float* dpos, int batch, int S, int C,
                                     int vocab, b200sd_stream_t stream) {
    B200SD_REQUIRE(ids && dx && dtok && dpos, "clip_embed_bwd: null pointer");
    B200SD_REQUIRE(batch > 0 && S > 0 && C > 0 && vocab > 0, "clip_embed_bwd: bad sizes");
    clip_embed_bwd_kernel<<<dim3(S), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(ids, dx, dtok, dpos,
                              batch, S, C, vocab);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_quick_gelu_fwd(const void* u, void* out, int64_t n, b200sd_stream_t stream) {
    B200SD_REQUIRE(u && out && n > 0 && n % 8 == 0, "quick_gelu_fwd: bad arguments (n must be a multiple of 8)");
    quick_gelu_fwd_kernel<<<dim3(ew_grid(n / 8, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(u), static_cast<bf16*>(out), n / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_quick_gelu_bwd(const void* u, const void* dg, void* du, int64_t n, b200sd_stream_t stream) {
    B200SD_REQUIRE(u && dg && du && n > 0 && n % 8 == 0, "quick_gelu_bwd: bad arguments (n must be a multiple of 8)");
    quick_gelu_bwd_kernel<<<dim3(ew_grid(n / 8, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(u), static_cast<const bf16*>(dg), static_cast<bf16*>(du), n / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_layernorm_f32out(const float* x, const float* gamma, const float* beta, float* out, int rows, int C, float eps,
                                       b200sd_stream_t stream) {
    B200SD_REQUIRE(x && gamma && beta && out && rows > 0 && C > 0, "layernorm_f32out: bad arguments");
    layernorm_f32out_kernel<<<dim3(ceil_div(rows, 8)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x,
                              gamma, beta, out, rows, C, eps);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

static int check_attn(int batch, int heads, int S, int d, int ld) {
    B200SD_REQUIRE(batch > 0 && heads > 0, "causal_attention: bad batch / heads");
    B200SD_REQUIRE(S >= 1 && S <= kMaxS, "causal_attention: S=%d unsupported (<= %d tokens)", S, kMaxS);
    B200SD_REQUIRE(d >= 8 && d <= kMaxD && d % 8 == 0, "causal_attention: head dim %d unsupported (multiple of 8, <= %d)", d, kMaxD);
    B200SD_REQUIRE(ld % 8 == 0, "causal_attention: leading dimension must be a multiple of 8 elements");
    return B200SD_OK;
}

extern "C" int b200sd_causal_attention(const void* qkv, void* out, int batch, int heads, int S, int d, int ld, int ldo, int q_off,
                                       int k_off, int v_off, float scale, b200sd_stream_t stream) {
    B200SD_REQUIRE(qkv && out, "causal_attention: null pointer");
    if (int rc = check_attn(batch, heads, S, d, ld)) return rc;
    B200SD_REQUIRE(q_off % 8 == 0 && k_off % 8 == 0 && v_off % 8 == 0, "causal_attention: offsets must be multiples of 8 elements");
    const size_t smem = (size_t)(3 * kMaxS * (kMaxD + 1) + kMaxS * (kMaxS + 1)) * sizeof(float);
    B200SD_CUDA(b200sd_opt_in_smem(clip_attention_fwd_kernel, (int)smem));
    clip_attention_fwd_kernel<<<dim3(heads, batch), dim3(256), smem, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(qkv), static_cast<bf16*>(out), S, d, ld, ldo, q_off, k_off, v_off, scale);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_causal_attention_bwd(const void* qkv, const void* dout, void* dqkv, int batch, int heads, int S, int d, int ld,
                                           int lddo, int ldd, int q_off, int k_off, int v_off, float scale, b200sd_stream_t stream) {
    B200SD_REQUIRE(qkv && dout && dqkv, "causal_attention_bwd: null pointer");
    if (int rc = check_attn(batch, heads, S, d, ld)) return rc;
    B200SD_REQUIRE(lddo % 8 == 0, "causal_attention_bwd: lddo must be a multiple of 8 elements");
    const size_t smem = (size_t)(4 * kMaxS * (kMaxD + 1) + 2 * kMaxS * (kMaxS + 1)) * sizeof(float);
    B200SD_CUDA(b200sd_opt_in_smem(clip_attention_bwd_kernel, (int)smem));
    clip_attention_bwd_kernel<<<dim3(heads, batch), dim3(256), smem, static_cast<cudaStream_t>(stream)>>>(
                              static_cast<const bf16*>(qkv), static_cast<const bf16*>(dout), static_cast<bf16*>(dqkv), S, d, ld, lddo,
                              ldd, q_off, k_off, v_off, scale);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
