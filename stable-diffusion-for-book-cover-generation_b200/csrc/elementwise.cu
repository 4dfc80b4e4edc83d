// b200sd -- scheduler / loss elementwise kernels (SURVEY.md K10-K13).  HBM-bound: 128-bit
// vectorised, coalesced, grid sized in multiples of the SM count.
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

constexpr int kThreads = 256;

template <int DT>
struct Elem;
template <>
struct Elem<B200SD_F32> {
    using T = float;
};
template <>
struct Elem<B200SD_BF16> {
    using T = bf16;
};

// 8 consecutive elements -> float[8]
template <int DT>
__device__ __forceinline__ void load8(const void* p, int64_t i, float (&v)[8]) {
    if constexpr (DT == B200SD_F32) {
        const float4* q = reinterpret_cast<const float4*>(static_cast<const float*>(p) + i);
        float4 a = __ldg(q), b = __ldg(q + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
        uint4 u = __ldg(reinterpret_cast<const uint4*>(static_cast<const bf16*>(p) + i));
        float2 f;
        f = unpack_bf16x2(u.x); v[0] = f.x; v[1] = f.y;
        f = unpack_bf16x2(u.y); v[2] = f.x; v[3] = f.y;
        f = unpack_bf16x2(u.z); v[4] = f.x; v[5] = f.y;
        f = unpack_bf16x2(u.w); v[6] = f.x; v[7] = f.y;
    }
}
template <int DT>
__device__ __forceinline__ void store8(void* p, int64_t i, const float (&v)[8]) {
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
template <int DT>
__device__ __forceinline__ float load1(const void* p, int64_t i) {
    if constexpr (DT == B200SD_F32) return static_cast<const float*>(p)[i];
    else return __bfloat162float(static_cast<const bf16*>(p)[i]);
}
template <int DT>
__device__ __forceinline__ void store1(void* p, int64_t i, float v) {
    if constexpr (DT == B200SD_F32) static_cast<float*>(p)[i] = v;
    else static_cast<bf16*>(p)[i] = __float2bfloat16_rn(v);
}

inline int grid_for(int64_t nvec) {
    int64_t blocks = (nvec + kThreads - 1) / kThreads;
    int64_t cap = (int64_t)b200sd_num_sms() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

// ---------------------------------------------------------------------------------------------
// CFG + PLMS
// ---------------------------------------------------------------------------------------------
struct PlmsArgs {
    const void* hist[4];
    float w[5];
    int nhist;
    float g, cx, ce;
};

template <int EDT, int XDT>
__global__ void __launch_bounds__(kThreads) cfg_plms_kernel(const void* __restrict__ eps_u,
                                                            const void* __restrict__ eps_c,
                                                            const void* __restrict__ x, void* __restrict__ out,
                                                            void* __restrict__ eps_out, int64_t n, int64_t nvec, PlmsArgs a) {
    const bool cfg = eps_c != nullptr;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float eu[8], ec[8], xv[8], e[8], acc[8], o[8];
        load8<EDT>(eps_u, i * 8, eu);
        if (cfg) load8<EDT>(eps_c, i * 8, ec);
        load8<XDT>(x, i * 8, xv);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            e[j] = cfg ? (eu[j] + a.g * (ec[j] - eu[j])) : eu[j];
            acc[j] = a.w[0] * e[j];
        }
        for (int h = 0; h < a.nhist; ++h) {
            float hv[8];
            load8<EDT>(a.hist[h], i * 8, hv);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += a.w[1 + h] * hv[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = a.cx * xv[j] - a.ce * acc[j];
        store8<XDT>(out, i * 8, o);
        if (eps_out) store8<EDT>(eps_out, i * 8, e);
    }
    {
        for (int64_t i = nvec * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            float eu = load1<EDT>(eps_u, i);
            float e = cfg ? (eu + a.g * (load1<EDT>(eps_c, i) - eu)) : eu;
            float acc = a.w[0] * e;
            for (int h = 0; h < a.nhist; ++h) acc += a.w[1 + h] * load1<EDT>(a.hist[h], i);
            store1<XDT>(out, i, a.cx * load1<XDT>(x, i) - a.ce * acc);
            if (eps_out) store1<EDT>(eps_out, i, e);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// add_noise
// ---------------------------------------------------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(kThreads) add_noise_kernel(const void* __restrict__ x0,
                                                             const void* __restrict__ noise,
                                                             const int64_t* __restrict__ timesteps,
                                                             const float* __restrict__ sa_table,
                                                             const float* __restrict__ sb_table,
                                                             void* __restrict__ out, int64_t per_sample, int64_t nvec, int T) {
    const int b = blockIdx.y;
    int64_t t = timesteps[b];
    t = t < 0 ? 0 : (t >= T ? T - 1 : t);
    const float sa = __ldg(sa_table + t), sb = __ldg(sb_table + t);
    const int64_t base = (int64_t)b * per_sample;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float a[8], e[8], o[8];
        load8<DT>(x0, base + i * 8, a);
        load8<DT>(noise, base + i * 8, e);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = sa * a[j] + sb * e[j];
        store8<DT>(out, base + i * 8, o);
    }
    {
        for (int64_t i = nvec * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_sample; i += stride)
            store1<DT>(out, base + i, sa * load1<DT>(x0, base + i) + sb * load1<DT>(noise, base + i));
    }
}

// ---------------------------------------------------------------------------------------------
// MSE
// ---------------------------------------------------------------------------------------------
constexpr int kMsePartials = 1024;

__device__ __forceinline__ float block_sum(float v, float* sm) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    float r = 0.f;
    if (warp == 0) {
        r = lane < (blockDim.x >> 5) ? sm[lane] : 0.f;
        r = warp_sum(r);
    }
    return r;  // valid in warp 0
}

template <int PDT, int TDT>
__global__ void __launch_bounds__(kThreads) mse_fwd_kernel(const void* __restrict__ pred,
                                                           const void* __restrict__ target,
                                                           float* __restrict__ loss_out, float* __restrict__ ws,
                                                           int64_t n, int64_t nvec) {
    __shared__ float sm[32];
    __shared__ bool is_last;
    float acc = 0.f;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float p[8], t[8];
        load8<PDT>(pred, i * 8, p);
        load8<TDT>(target, i * 8, t);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float d = p[j] - t[j];
            acc += d * d;
        }
    }
    {
        for (int64_t i = nvec * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            float d = load1<PDT>(pred, i) - load1<TDT>(target, i);
            acc += d * d;
        }
    }
    float bs = block_sum(acc, sm);
    unsigned int* counter = reinterpret_cast<unsigned int*>(ws + kMsePartials);
    if (threadIdx.x == 0) {
        ws[blockIdx.x] = bs;
        __threadfence();
        unsigned int prev = atomicAdd(counter, 1u);
        is_last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        // deterministic: fixed-order tree over the per-block partials, accumulated in double
        double s = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) s += (double)__ldcg(ws + i);
        __shared__ double dsm[kThreads];
        dsm[threadIdx.x] = s;
        __syncthreads();
        for (int o = kThreads / 2; o > 0; o >>= 1) {
            if (threadIdx.x < o) dsm[threadIdx.x] += dsm[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            loss_out[0] = (float)(dsm[0] / (double)n);
            *counter = 0;  // self-cleaning for the next launch
        }
    }
}

template <int PDT, int TDT>
__global__ void __launch_bounds__(kThreads) mse_bwd_kernel(const void* __restrict__ pred,
                                                           const void* __restrict__ target,
                                                           const float* __restrict__ grad_loss,
                                                           void* __restrict__ grad_pred, int64_t n, int64_t nvec) {
    const float s = __ldg(grad_loss) * 2.0f / (float)n;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float p[8], t[8], g[8];
        load8<PDT>(pred, i * 8, p);
        load8<TDT>(target, i * 8, t);
#pragma unroll
        for (int j = 0; j < 8; ++j) g[j] = s * (p[j] - t[j]);
        store8<PDT>(grad_pred, i * 8, g);
    }
    {
        for (int64_t i = nvec * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
            store1<PDT>(grad_pred, i, s * (load1<PDT>(pred, i) - load1<TDT>(target, i)));
    }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

#define DISPATCH2(E, X, KERNEL, GRID, STREAM, ...)                                                    \
    do {                                                                                              \
        if ((E) == B200SD_F32 && (X) == B200SD_F32)                                                   \
            KERNEL<B200SD_F32, B200SD_F32><<<dim3(GRID), dim3(kThreads), 0, STREAM>>>(__VA_ARGS__);   \
        else if ((E) == B200SD_BF16 && (X) == B200SD_F32)                                             \
            KERNEL<B200SD_BF16, B200SD_F32><<<dim3(GRID), dim3(kThreads), 0, STREAM>>>(__VA_ARGS__);  \
        else if ((E) == B200SD_F32 && (X) == B200SD_BF16)                                             \
            KERNEL<B200SD_F32, B200SD_BF16><<<dim3(GRID), dim3(kThreads), 0, STREAM>>>(__VA_ARGS__);  \
        else                                                                                          \
            KERNEL<B200SD_BF16, B200SD_BF16><<<dim3(GRID), dim3(kThreads), 0, STREAM>>>(__VA_ARGS__); \
    } while (0)

static bool dtype_ok(int d) { return d == B200SD_F32 || d == B200SD_BF16; }

// Captured sampler (one CUDA graph per denoising step, replayed with no host-side arguments): the step index lives on the
// device.  cursor[0] = next step, cursor[1] = the step being executed.
namespace {
__global__ void sampler_advance_kernel(const float* __restrict__ timesteps, int n_steps, int* __restrict__ cursor,
                                       float* __restrict__ in_t, int n_t) {
    const int c = cursor[0];
    const float t = timesteps[c];
    for (int i = threadIdx.x; i < n_t; i += blockDim.x) in_t[i] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        cursor[1] = c;
        cursor[0] = (c + 1 == n_steps) ? 0 : c + 1;
    }
}
}  // namespace

extern "C" int b200sd_sampler_advance(const float* timesteps, int n_steps, int* cursor, float* in_t, int n_t,
                                      b200sd_stream_t stream) {
    B200SD_REQUIRE(timesteps && cursor && in_t, "sampler_advance: null pointer");
    B200SD_REQUIRE(n_steps > 0 && n_t > 0, "sampler_advance: empty table");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    sampler_advance_kernel<<<dim3(1), dim3(64), 0, s>>>(timesteps, n_steps, cursor, in_t, n_t);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// Captured PLMS step: everything that changes from call to call -- the linear-multistep weights, which slots of the 4-deep eps
// ring hold the history, where this call's eps goes, whether x is the running sample or the one saved by the first call
// (PNDM's second call re-does the first timestep), the two scalars of _get_prev_sample -- is one row of a device table indexed
// by the cursor.  Row layout (12 floats): w0 w1 w2 w3 | cx ce | h1 h2 h3 (ring slots, -1 = unused) | out_slot (-1 = not
// kept) | x_from_saved | save_x.
namespace {
constexpr int kPlmsRow = 12;
__global__ void __launch_bounds__(kThreads) cfg_plms_table_kernel(const float* __restrict__ eps_u, const float* __restrict__ eps_c,
                                                                  float* __restrict__ x, float* __restrict__ saved,
                                                                  float* __restrict__ ring, int64_t n, float g,
                                                                  const float* __restrict__ table, const int* __restrict__ cursor) {
    const float* row = table + (size_t)cursor[1] * kPlmsRow;
    const float w0 = row[0], w1 = row[1], w2 = row[2], w3 = row[3], cx = row[4], ce = row[5];
    const int h1 = (int)row[6], h2 = (int)row[7], h3 = (int)row[8], slot = (int)row[9];
    const bool from_saved = row[10] != 0.f, save_x = row[11] != 0.f;
    const bool cfg = eps_c != nullptr;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float eu = eps_u[i];
        const float e = cfg ? (eu + g * (eps_c[i] - eu)) : eu;
        float acc = w0 * e;
        if (h1 >= 0) acc = fmaf(w1, ring[(size_t)h1 * n + i], acc);
        if (h2 >= 0) acc = fmaf(w2, ring[(size_t)h2 * n + i], acc);
        if (h3 >= 0) acc = fmaf(w3, ring[(size_t)h3 * n + i], acc);
        const float cur = x[i];
        const float xv = from_saved ? saved[i] : cur;
        if (save_x) saved[i] = cur;
        x[i] = cx * xv - ce * acc;
        if (slot >= 0) ring[(size_t)slot * n + i] = e;
    }
}
}  // namespace

extern "C" int b200sd_cfg_plms_step_table(const float* eps_u, const float* eps_c, float* x, float* saved, float* ring, int64_t n,
                                          float guidance, const float* table, const int* cursor, b200sd_stream_t stream) {
    B200SD_REQUIRE(eps_u && x && saved && ring && table && cursor, "cfg_plms_step_table: null pointer");
    B200SD_REQUIRE(n >= 0, "cfg_plms_step_table: negative n");
    if (n == 0) return B200SD_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cfg_plms_table_kernel<<<dim3(grid_for(n)), dim3(kThreads), 0, s>>>(eps_u, eps_c, x, saved, ring, n, guidance,
                              table, cursor);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// DDIM (eta = 0 is c_x0 = sqrt(abar_prev), c_x = 0, c_e = sqrt(1 - abar_prev), no noise; eta > 0 adds sigma z) and DDPM:
// the DDIM prediction of x0, then
//   x' = c_x0 x0 + c_x x + c_e eps + c_z z
// z ~ N(0, 1) is drawn by the host from the caller's torch.Generator, so the per-call and the captured loop consume the same
// noise.  Table row (8 floats): sa_t sb_t c_x0 c_x c_e c_z noise_row clip; noise_row = -1: no noise term, z is not read.
namespace {
constexpr int kAncestralRow = 8;

struct AncestralCoef {
    float g, sa_t, sb_t, c_x0, c_x, c_e, c_z;
    bool clip;
};

__device__ __forceinline__ float ancestral_one(float eu, float ec, float x, float z, bool cfg, bool has_z,
                                               const AncestralCoef& c) {
    const float e = cfg ? (eu + c.g * (ec - eu)) : eu;
    float x0 = (x - c.sb_t * e) / c.sa_t;
    if (c.clip) x0 = fminf(fmaxf(x0, -1.f), 1.f);
    const float mean = c.c_x0 * x0 + c.c_x * x + c.c_e * e;
    return has_z ? mean + c.c_z * z : mean;
}

// x and out may alias (the table form updates the latents in place): each element is read before it is written, by the
// same thread.
template <int EDT, int XDT>
__global__ void __launch_bounds__(kThreads) cfg_ancestral_kernel(const void* __restrict__ eps_u,
                                                                 const void* __restrict__ eps_c, const void* x,
                                                                 const float* __restrict__ noise, void* out, int64_t n,
                                                                 int64_t nvec, AncestralCoef c,
                                                                 const float* __restrict__ table,
                                                                 const int* __restrict__ cursor) {
    if (table != nullptr) {
        const float4* row = reinterpret_cast<const float4*>(table + (size_t)cursor[1] * kAncestralRow);
        const float4 a = row[0], b = row[1];
        c.sa_t = a.x, c.sb_t = a.y, c.c_x0 = a.z, c.c_x = a.w, c.c_e = b.x, c.c_z = b.y;
        const int noise_row = (int)b.z;
        noise = (noise_row < 0 || noise == nullptr) ? nullptr : noise + (size_t)noise_row * n;
        c.clip = b.w != 0.f;
    }
    const bool cfg = eps_c != nullptr, has_z = noise != nullptr;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float eu[8], ec[8], xv[8], z[8] = {}, o[8];
        load8<EDT>(eps_u, i * 8, eu);
        if (cfg) load8<EDT>(eps_c, i * 8, ec);
        load8<XDT>(x, i * 8, xv);
        if (has_z) load8<B200SD_F32>(noise, i * 8, z);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = ancestral_one(eu[j], ec[j], xv[j], z[j], cfg, has_z, c);
        store8<XDT>(out, i * 8, o);
    }
    for (int64_t i = nvec * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float eu = load1<EDT>(eps_u, i);
        const float ec = cfg ? load1<EDT>(eps_c, i) : 0.f;
        const float z = has_z ? noise[i] : 0.f;
        store1<XDT>(out, i, ancestral_one(eu, ec, load1<XDT>(x, i), z, cfg, has_z, c));
    }
}
}  // namespace

extern "C" int b200sd_cfg_ancestral_step(const void* eps_u, const void* eps_c, const void* x, const float* noise, void* out,
                                         int64_t n, float guidance, float sa_t, float sb_t, float c_x0, float c_x, float c_e,
                                         float c_z, int clip, int eps_dtype, int x_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(eps_u && x && out, "cfg_ancestral_step: null pointer");
    B200SD_REQUIRE(n >= 0, "cfg_ancestral_step: negative n");
    B200SD_REQUIRE(dtype_ok(eps_dtype) && dtype_ok(x_dtype), "cfg_ancestral_step: bad dtype");
    B200SD_REQUIRE(sa_t != 0.f, "cfg_ancestral_step: sa_t == 0");
    const bool vec = aligned16(eps_u) && aligned16(eps_c) && aligned16(x) && aligned16(noise) && aligned16(out);
    const int64_t nvec = vec ? n / 8 : 0;  // unaligned views take the scalar path
    if (n == 0) return B200SD_OK;
    AncestralCoef c{guidance, sa_t, sb_t, c_x0, c_x, c_e, c_z, clip != 0};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH2(eps_dtype, x_dtype, cfg_ancestral_kernel, grid_for(vec ? n / 8 : n), s, eps_u, eps_c, x, noise, out, n, nvec, c,
              (const float*)nullptr, (const int*)nullptr);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_cfg_ddim_step(const void* eps_u, const void* eps_c, const void* x, void* out, void* eps_out,
                                    int64_t n, float guidance, float sa_t, float sb_t, float sa_p, float sb_p,
                                    int eps_dtype, int x_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(eps_out == nullptr, "cfg_ddim_step: eps_out is no longer supported and must be NULL");
    return b200sd_cfg_ancestral_step(eps_u, eps_c, x, nullptr, out, n, guidance, sa_t, sb_t, sa_p, 0.f, sb_p, 0.f, 0, eps_dtype,
                                     x_dtype, stream);
}

extern "C" int b200sd_cfg_ancestral_step_table(const float* eps_u, const float* eps_c, float* x, const float* noise, int64_t n,
                                               float guidance, const float* table, const int* cursor, b200sd_stream_t stream) {
    B200SD_REQUIRE(eps_u && x && table && cursor, "cfg_ancestral_step_table: null pointer");
    B200SD_REQUIRE(n >= 0, "cfg_ancestral_step_table: negative n");
    B200SD_REQUIRE(aligned16(table), "cfg_ancestral_step_table: table must be 16-byte aligned");
    // every noise row must be 16-byte aligned for the vector path: the base pointer and the row pitch n
    const bool vec = aligned16(eps_u) && aligned16(eps_c) && aligned16(x) && aligned16(noise) && n % 4 == 0;
    const int64_t nvec = vec ? n / 8 : 0;
    if (n == 0) return B200SD_OK;
    AncestralCoef c{guidance, 1.f, 0.f, 1.f, 0.f, 0.f, 0.f, false};
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cfg_ancestral_kernel<B200SD_F32, B200SD_F32><<<dim3(grid_for(vec ? n / 8 : n)), dim3(kThreads), 0, s>>>(
        eps_u, eps_c, x, noise, x, n, nvec, c, table, cursor);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_cfg_plms_step(const void* eps_u, const void* eps_c, const void* x, void* out, void* eps_out,
                                    const void* hist0, const void* hist1, const void* hist2, const void* hist3,
                                    int nhist, const float* w_host5, int64_t n, float guidance, float cx, float ce,
                                    int eps_dtype, int x_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(eps_u && x && out && w_host5, "cfg_plms_step: null pointer");
    B200SD_REQUIRE(nhist >= 0 && nhist <= 4, "cfg_plms_step: nhist out of range");
    B200SD_REQUIRE(dtype_ok(eps_dtype) && dtype_ok(x_dtype), "cfg_plms_step: bad dtype");
    PlmsArgs a;
    a.hist[0] = hist0; a.hist[1] = hist1; a.hist[2] = hist2; a.hist[3] = hist3;
    bool vec = aligned16(eps_u) && aligned16(eps_c) && aligned16(x) && aligned16(out) && aligned16(eps_out);
    for (int i = 0; i < nhist; ++i) {
        B200SD_REQUIRE(a.hist[i] != nullptr, "cfg_plms_step: null history pointer");
        vec = vec && aligned16(a.hist[i]);
    }
    const int64_t nvec = vec ? n / 8 : 0;
    for (int i = 0; i < 5; ++i) a.w[i] = w_host5[i];
    a.nhist = nhist; a.g = guidance; a.cx = cx; a.ce = ce;
    if (n == 0) return B200SD_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH2(eps_dtype, x_dtype, cfg_plms_kernel, grid_for(vec ? n / 8 : n), s, eps_u, eps_c, x, out, eps_out, n, nvec, a);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_add_noise(const void* x0, const void* noise, const int64_t* timesteps, const float* sa_table,
                                const float* sb_table, void* out, int batch, int64_t per_sample,
                                int num_train_timesteps, int dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(x0 && noise && timesteps && sa_table && sb_table && out, "add_noise: null pointer");
    B200SD_REQUIRE(batch >= 0 && per_sample >= 0 && batch <= 65535, "add_noise: bad sizes");
    B200SD_REQUIRE(dtype_ok(dtype), "add_noise: bad dtype");
    const bool vec = aligned16(x0) && aligned16(noise) && aligned16(out) && (per_sample % 8 == 0 || batch <= 1);
    const int64_t nvec = vec ? per_sample / 8 : 0;
    if (batch == 0 || per_sample == 0) return B200SD_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int gx = grid_for(vec ? per_sample / 8 : per_sample);
    int cap = b200sd_num_sms() * 8 / batch;
    if (cap < 1) cap = 1;
    if (gx > cap) gx = cap;
    dim3 grid(gx, batch);
    if (dtype == B200SD_F32)
        add_noise_kernel<B200SD_F32><<<dim3(grid), dim3(kThreads), 0, s>>>(x0, noise, timesteps, sa_table, sb_table, out, per_sample, nvec, num_train_timesteps);
    else
        add_noise_kernel<B200SD_BF16><<<dim3(grid), dim3(kThreads), 0, s>>>(x0, noise, timesteps, sa_table, sb_table, out, per_sample, nvec, num_train_timesteps);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// Legacy inpainting (diffusers 0.7.2 StableDiffusionInpaintPipelineLegacy), after every scheduler step at loop timestep t:
//   x <- m (sa[t] x0 + sb[t] z) + (1 - m) x
// i.e. the kept region is re-noised from the original latents with the same noise every step.  m, x0, z have x's full shape
// (the host expands the mask).  The timestep comes by value or, in the captured sampler, from t_table[cursor[1]].
namespace {
__global__ void __launch_bounds__(kThreads) inpaint_blend_kernel(float* x, const float* __restrict__ x0,
                                                                 const float* __restrict__ z, const float* __restrict__ m,
                                                                 const float* __restrict__ sa_table,
                                                                 const float* __restrict__ sb_table, int T, int64_t t,
                                                                 const float* __restrict__ t_table,
                                                                 const int* __restrict__ cursor, int64_t n, int64_t nvec) {
    if (t_table != nullptr) t = (int64_t)t_table[cursor[1]];
    t = t < 0 ? 0 : (t >= T ? T - 1 : t);
    const float sa = __ldg(sa_table + t), sb = __ldg(sb_table + t);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float xv[8], a[8], e[8], mv[8], o[8];
        load8<B200SD_F32>(x, i * 8, xv);
        load8<B200SD_F32>(x0, i * 8, a);
        load8<B200SD_F32>(z, i * 8, e);
        load8<B200SD_F32>(m, i * 8, mv);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = mv[j] * (sa * a[j] + sb * e[j]) + (1.f - mv[j]) * xv[j];
        store8<B200SD_F32>(x, i * 8, o);
    }
    for (int64_t i = nvec * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        x[i] = m[i] * (sa * x0[i] + sb * z[i]) + (1.f - m[i]) * x[i];
}

int inpaint_blend_launch(float* x, const float* x0, const float* noise, const float* mask, int64_t n, int64_t timestep,
                         const float* t_table, const int* cursor, const float* sa_table, const float* sb_table,
                         int num_train_timesteps, b200sd_stream_t stream) {
    B200SD_REQUIRE(x && x0 && noise && mask && sa_table && sb_table, "inpaint_blend: null pointer");
    B200SD_REQUIRE(n >= 0 && num_train_timesteps > 0, "inpaint_blend: bad sizes");
    const bool vec = aligned16(x) && aligned16(x0) && aligned16(noise) && aligned16(mask);
    const int64_t nvec = vec ? n / 8 : 0;
    if (n == 0) return B200SD_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    inpaint_blend_kernel<<<dim3(grid_for(vec ? n / 8 : n)), dim3(kThreads), 0, s>>>(
        x, x0, noise, mask, sa_table, sb_table, num_train_timesteps, timestep, t_table, cursor, n, nvec);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
}  // namespace

extern "C" int b200sd_inpaint_blend(float* x, const float* x0, const float* noise, const float* mask, int64_t n,
                                    int64_t timestep, const float* sa_table, const float* sb_table, int num_train_timesteps,
                                    b200sd_stream_t stream) {
    return inpaint_blend_launch(x, x0, noise, mask, n, timestep, nullptr, nullptr, sa_table, sb_table, num_train_timesteps,
                                stream);
}

extern "C" int b200sd_inpaint_blend_table(float* x, const float* x0, const float* noise, const float* mask, int64_t n,
                                          const float* t_table, const int* cursor, const float* sa_table, const float* sb_table,
                                          int num_train_timesteps, b200sd_stream_t stream) {
    B200SD_REQUIRE(t_table && cursor, "inpaint_blend_table: null pointer");
    return inpaint_blend_launch(x, x0, noise, mask, n, 0, t_table, cursor, sa_table, sb_table, num_train_timesteps, stream);
}

extern "C" int b200sd_mse_workspace_floats(void) { return kMsePartials + 4; }

extern "C" int b200sd_mse_loss_fwd(const void* pred, const void* target, float* loss_out, float* workspace,
                                   int64_t n, int pred_dtype, int target_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(pred && target && loss_out && workspace, "mse_loss_fwd: null pointer");
    B200SD_REQUIRE(n > 0, "mse_loss_fwd: n must be positive");
    B200SD_REQUIRE(dtype_ok(pred_dtype) && dtype_ok(target_dtype), "mse_loss_fwd: bad dtype");
    const bool vec = aligned16(pred) && aligned16(target);
    const int64_t nvec = vec ? n / 8 : 0;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int grid = grid_for(vec ? n / 8 : n);
    if (grid > kMsePartials) grid = kMsePartials;
    DISPATCH2(pred_dtype, target_dtype, mse_fwd_kernel, grid, s, pred, target, loss_out, workspace, n, nvec);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_mse_loss_bwd(const void* pred, const void* target, const float* grad_loss, void* grad_pred,
                                   int64_t n, int pred_dtype, int target_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(pred && target && grad_loss && grad_pred, "mse_loss_bwd: null pointer");
    B200SD_REQUIRE(n > 0, "mse_loss_bwd: n must be positive");
    B200SD_REQUIRE(dtype_ok(pred_dtype) && dtype_ok(target_dtype), "mse_loss_bwd: bad dtype");
    const bool vec = aligned16(pred) && aligned16(target) && aligned16(grad_pred);
    const int64_t nvec = vec ? n / 8 : 0;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH2(pred_dtype, target_dtype, mse_bwd_kernel, grid_for(vec ? n / 8 : n), s, pred, target, grad_loss, grad_pred, n, nvec);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
