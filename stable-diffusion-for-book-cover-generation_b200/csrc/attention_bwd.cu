// b200sd -- backward of the fused attention (autograd through CrossAttention._attention, SURVEY.md rows A5/A9).
//
//   P = softmax(scale Q K^T) (recomputed from the saved log-sum-exp, never materialised in HBM)
//   dV = P^T dO ;  dP = dO V^T ;  dS = P o (dP - delta) * scale,  delta = rowsum(dO o O)
//   dQ = dS K  ;  dK = dS^T Q
//
// Two deterministic kernels (no atomics): `attn_bwd_dq_kernel` owns 64 query rows and streams key tiles;
// `attn_bwd_dkv_kernel` owns 64 keys and streams query tiles.  Both use warp-level tensor-core MMA
// (mma.sync m16n8k16 bf16, fp32 accumulate) with cp.async double-buffered tiles, like the register-resident
// forward kernel in attention.cu; head dims 40 / 80 / 160 are zero-padded to a multiple of 16 in shared memory.
// For head dims > 96 the dK/dV accumulators are split in two halves of d across CTAs (register budget).
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

constexpr int kT = 64;          // rows per tile (queries and keys)
constexpr int kThreads = 128;   // 4 warps x 16 rows

__device__ __forceinline__ void cp_async16(void* dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ptx::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src, int src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(ptx::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(ptx::smem_u32(p)));
}
__device__ __forceinline__ void ldsm4t(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(ptx::smem_u32(p)));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows x chunks 16-byte pieces, global [row][ld] -> smem [row][PITCH]; rows >= valid are zero-filled
template <int PITCH>
__device__ __forceinline__ void load_rows(uint8_t* smem, const bf16* g, int ld, int valid, int chunks) {
    for (int i = threadIdx.x; i < kT * chunks; i += kThreads) {
        const int r = i / chunks, c = i % chunks;
        const bool ok = r < valid;
        cp_async16(smem + (size_t)r * PITCH + c * 16, g + (size_t)(ok ? r : 0) * ld + c * 8, ok ? 16 : 0);
    }
}
// one fp32 per row; rows >= valid get `fill` written directly (cp.async zero-fill cannot produce +inf)
__device__ __forceinline__ void load_vec(float* smem, const float* g, int valid, float fill) {
    if (threadIdx.x < kT) {
        if (threadIdx.x < valid) cp_async4(smem + threadIdx.x, g + threadIdx.x, 4);
        else smem[threadIdx.x] = fill;
    }
}
template <int PITCH>
__device__ __forceinline__ void zero_pad(uint8_t* smem, int rows, int chunks) {
    constexpr int SLOTS = PITCH / 16;
    for (int i = threadIdx.x; i < rows * (SLOTS - chunks); i += kThreads) {
        const int r = i / (SLOTS - chunks), c = chunks + i % (SLOTS - chunks);
        *reinterpret_cast<uint4*>(smem + (size_t)r * PITCH + c * 16) = make_uint4(0, 0, 0, 0);
    }
}

// C[16 x 64] = A[16 x DP] * B^T, A rows = this warp's 16 rows of sA, B = 64 rows of sB, both [row][d] (K-major)
template <int DP, int PITCH>
__device__ __forceinline__ void mma_rows_x_rowsT(float (&c)[8][4], const uint8_t* sA, const uint8_t* sB, int warp, int lane) {
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = c[i][2] = c[i][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < DP / 16; ++ks) {
        uint32_t a[4];
        ldsm4(a, sA + (size_t)(warp * 16 + (lane & 15)) * PITCH + (ks * 16 + (lane >> 4) * 8) * 2);
#pragma unroll
        for (int np = 0; np < 4; ++np) {
            uint32_t b[4];
            ldsm4(b, sB + (size_t)(np * 16 + (lane & 7) + (lane >> 4) * 8) * PITCH + (ks * 16 + ((lane >> 3) & 1) * 8) * 2);
            mma16816(c[2 * np], a, b[0], b[1]);
            mma16816(c[2 * np + 1], a, b[2], b[3]);
        }
    }
}
// acc[16 x (16*NKS)] += A[16 x 64] * B[64 x d-range], A from fp32 accumulators `s`, B = sB [64 rows][d] read transposed
template <int NKS, int PITCH>
__device__ __forceinline__ void mma_acc_x_rows(float (&acc)[2 * NKS][4], const float (&s)[8][4], const uint8_t* sB, int d0, int lane) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        uint32_t a[4];
        a[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
        a[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
        a[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        a[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int dp = 0; dp < NKS; ++dp) {
            uint32_t b[4];
            ldsm4t(b, sB + (size_t)(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * PITCH + (d0 + dp * 16 + (lane >> 4) * 8) * 2);
            mma16816(acc[2 * dp], a, b[0], b[1]);
            mma16816(acc[2 * dp + 1], a, b[2], b[3]);
        }
    }
}

struct BwdParams {
    const bf16 *q, *k, *v, *dout;
    const float *lse, *delta;
    bf16 *dq, *dk, *dv;
    int Sq, Skv, D, heads;
    int ldq, ldk, ldv, ldo, lddq, lddk, lddv;
    float scale, scale_log2;
};

// ---- delta[b, h, row] = sum_d dO o O -------------------------------------------------------------------------
__global__ void attn_delta_kernel(const bf16* __restrict__ o, const bf16* __restrict__ dout, float* __restrict__ delta,
                                  int batch, int heads, int Sq, int D, int ldo, int lddo) {
    const int64_t total = (int64_t)batch * Sq * heads;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(i % heads);
        const int64_t row = i / heads;
        float a = 0.f;
        for (int c = 0; c < D; c += 8) {
            float x[8], y[8];
            ld8<B200SD_BF16>(o, (size_t)row * ldo + h * D + c, x);
            ld8<B200SD_BF16>(dout, (size_t)row * lddo + h * D + c, y);
#pragma unroll
            for (int j = 0; j < 8; ++j) a += x[j] * y[j];
        }
        const int b = (int)(row / Sq), r = (int)(row % Sq);
        delta[((size_t)b * heads + h) * Sq + r] = a;
    }
}

// ---- dQ ------------------------------------------------------------------------------------------------------
template <int DP>
__global__ void __launch_bounds__(kThreads) attn_bwd_dq_kernel(const BwdParams p) {
    constexpr int PITCH = DP * 2 + 16;
    constexpr int KS = DP / 16;
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* sQ = smem;
    uint8_t* sdO = sQ + kT * PITCH;
    uint8_t* sK = sdO + kT * PITCH;        // [2]
    uint8_t* sV = sK + 2 * kT * PITCH;     // [2]
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * kT;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int D = p.D, chunks = D / 8;
    zero_pad<PITCH>(smem, 6 * kT, chunks);
    const bf16* qg = p.q + ((size_t)b * p.Sq + q0) * p.ldq + h * D;
    const bf16* dog = p.dout + ((size_t)b * p.Sq + q0) * p.ldo + h * D;
    const bf16* kg = p.k + (size_t)b * p.Skv * p.ldk + h * D;
    const bf16* vg = p.v + (size_t)b * p.Skv * p.ldv + h * D;
    const int qvalid = min(kT, p.Sq - q0);
    const int tiles = (p.Skv + kT - 1) / kT;
    load_rows<PITCH>(sQ, qg, p.ldq, qvalid, chunks);
    load_rows<PITCH>(sdO, dog, p.ldo, qvalid, chunks);
    load_rows<PITCH>(sK, kg, p.ldk, min(kT, p.Skv), chunks);
    load_rows<PITCH>(sV, vg, p.ldv, min(kT, p.Skv), chunks);
    cp_async_commit();

    const int r0 = q0 + warp * 16 + (lane >> 2), r1 = r0 + 8;
    const size_t vec_base = ((size_t)b * p.heads + h) * p.Sq;
    const float lse0 = r0 < p.Sq ? p.lse[vec_base + r0] : INFINITY, lse1 = r1 < p.Sq ? p.lse[vec_base + r1] : INFINITY;
    const float dl0 = r0 < p.Sq ? p.delta[vec_base + r0] : 0.f, dl1 = r1 < p.Sq ? p.delta[vec_base + r1] : 0.f;
    float acc[2 * KS][4];
#pragma unroll
    for (int i = 0; i < 2 * KS; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;

    for (int j = 0; j < tiles; ++j) {
        cp_async_wait_all();
        __syncthreads();
        if (j + 1 < tiles) {
            const int nb = (j + 1) & 1, valid = min(kT, p.Skv - (j + 1) * kT);
            load_rows<PITCH>(sK + (size_t)nb * kT * PITCH, kg + (size_t)(j + 1) * kT * p.ldk, p.ldk, valid, chunks);
            load_rows<PITCH>(sV + (size_t)nb * kT * PITCH, vg + (size_t)(j + 1) * kT * p.ldv, p.ldv, valid, chunks);
            cp_async_commit();
        }
        const uint8_t* tK = sK + (size_t)(j & 1) * kT * PITCH;
        const uint8_t* tV = sV + (size_t)(j & 1) * kT * PITCH;
        float s[8][4], dp[8][4];
        mma_rows_x_rowsT<DP, PITCH>(s, sQ, tK, warp, lane);
        mma_rows_x_rowsT<DP, PITCH>(dp, sdO, tV, warp, lane);
        const int kbase = j * kT;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int key = kbase + nt * 8 + (lane & 3) * 2;
            const bool ok0 = key < p.Skv, ok1 = key + 1 < p.Skv;
            const float p00 = ok0 ? exp2f(s[nt][0] * p.scale_log2 - lse0) : 0.f;
            const float p01 = ok1 ? exp2f(s[nt][1] * p.scale_log2 - lse0) : 0.f;
            const float p10 = ok0 ? exp2f(s[nt][2] * p.scale_log2 - lse1) : 0.f;
            const float p11 = ok1 ? exp2f(s[nt][3] * p.scale_log2 - lse1) : 0.f;
            s[nt][0] = p00 * (dp[nt][0] - dl0) * p.scale;
            s[nt][1] = p01 * (dp[nt][1] - dl0) * p.scale;
            s[nt][2] = p10 * (dp[nt][2] - dl1) * p.scale;
            s[nt][3] = p11 * (dp[nt][3] - dl1) * p.scale;
        }
        mma_acc_x_rows<KS, PITCH>(acc, s, tK, 0, lane);
    }
#pragma unroll
    for (int nt = 0; nt < 2 * KS; ++nt) {
        const int col = nt * 8 + (lane & 3) * 2;
        if (col < D) {
            if (r0 < p.Sq) *reinterpret_cast<uint32_t*>(p.dq + ((size_t)b * p.Sq + r0) * p.lddq + h * D + col) = pack_bf16x2(acc[nt][0], acc[nt][1]);
            if (r1 < p.Sq) *reinterpret_cast<uint32_t*>(p.dq + ((size_t)b * p.Sq + r1) * p.lddq + h * D + col) = pack_bf16x2(acc[nt][2], acc[nt][3]);
        }
    }
}

// ---- dK, dV --------------------------------------------------------------------------------------------------
// DSPLIT = number of CTAs sharing one key tile, each accumulating DP / DSPLIT columns of dK / dV
template <int DP, int DSPLIT>
__global__ void __launch_bounds__(kThreads) attn_bwd_dkv_kernel(const BwdParams p) {
    constexpr int PITCH = DP * 2 + 16;
    constexpr int NKS = DP / 16 / DSPLIT;   // 16-column blocks of the accumulators owned by this CTA
    static_assert((DP / 16) % DSPLIT == 0, "head-dim blocks must split evenly");
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* sK = smem;
    uint8_t* sV = sK + kT * PITCH;
    uint8_t* sQ = sV + kT * PITCH;          // [2]
    uint8_t* sdO = sQ + 2 * kT * PITCH;     // [2]
    float* sLse = reinterpret_cast<float*>(sdO + 2 * kT * PITCH);   // [2][64]
    float* sDel = sLse + 2 * kT;                                    // [2][64]
    const int b = blockIdx.z, h = blockIdx.y;
    const int kt = blockIdx.x / DSPLIT, dh = blockIdx.x % DSPLIT;
    const int k0 = kt * kT, d0 = dh * NKS * 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int D = p.D, chunks = D / 8;
    zero_pad<PITCH>(smem, 6 * kT, chunks);
    const bf16* kg = p.k + ((size_t)b * p.Skv + k0) * p.ldk + h * D;
    const bf16* vg = p.v + ((size_t)b * p.Skv + k0) * p.ldv + h * D;
    const bf16* qg = p.q + (size_t)b * p.Sq * p.ldq + h * D;
    const bf16* dog = p.dout + (size_t)b * p.Sq * p.ldo + h * D;
    const size_t vec_base = ((size_t)b * p.heads + h) * p.Sq;
    const int kvalid = min(kT, p.Skv - k0);
    const int tiles = (p.Sq + kT - 1) / kT;
    load_rows<PITCH>(sK, kg, p.ldk, kvalid, chunks);
    load_rows<PITCH>(sV, vg, p.ldv, kvalid, chunks);
    {
        const int valid = min(kT, p.Sq);
        load_rows<PITCH>(sQ, qg, p.ldq, valid, chunks);
        load_rows<PITCH>(sdO, dog, p.ldo, valid, chunks);
        load_vec(sLse, p.lse + vec_base, valid, INFINITY);
        load_vec(sDel, p.delta + vec_base, valid, 0.f);
    }
    cp_async_commit();

    float dk[2 * NKS][4], dv[2 * NKS][4];
#pragma unroll
    for (int i = 0; i < 2 * NKS; ++i) {
        dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
        dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
    }
    for (int j = 0; j < tiles; ++j) {
        cp_async_wait_all();
        __syncthreads();
        if (j + 1 < tiles) {
            const int nb = (j + 1) & 1, valid = min(kT, p.Sq - (j + 1) * kT);
            load_rows<PITCH>(sQ + (size_t)nb * kT * PITCH, qg + (size_t)(j + 1) * kT * p.ldq, p.ldq, valid, chunks);
            load_rows<PITCH>(sdO + (size_t)nb * kT * PITCH, dog + (size_t)(j + 1) * kT * p.ldo, p.ldo, valid, chunks);
            load_vec(sLse + nb * kT, p.lse + vec_base + (size_t)(j + 1) * kT, valid, INFINITY);
            load_vec(sDel + nb * kT, p.delta + vec_base + (size_t)(j + 1) * kT, valid, 0.f);
            cp_async_commit();
        }
        const uint8_t* tQ = sQ + (size_t)(j & 1) * kT * PITCH;
        const uint8_t* tdO = sdO + (size_t)(j & 1) * kT * PITCH;
        const float* tL = sLse + (j & 1) * kT;
        const float* tD = sDel + (j & 1) * kT;
        // S^T = K Q^T (16 keys x 64 queries per warp) -> P^T
        float s[8][4], dp[8][4];
        mma_rows_x_rowsT<DP, PITCH>(s, sK, tQ, warp, lane);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int qc = nt * 8 + (lane & 3) * 2;
            const float l0 = tL[qc], l1 = tL[qc + 1];
            s[nt][0] = exp2f(s[nt][0] * p.scale_log2 - l0);
            s[nt][1] = exp2f(s[nt][1] * p.scale_log2 - l1);
            s[nt][2] = exp2f(s[nt][2] * p.scale_log2 - l0);
            s[nt][3] = exp2f(s[nt][3] * p.scale_log2 - l1);
        }
        // dV += P^T dO
        mma_acc_x_rows<NKS, PITCH>(dv, s, tdO, d0, lane);
        // dP^T = V dO^T ; dS^T = P^T o (dP^T - delta) * scale
        mma_rows_x_rowsT<DP, PITCH>(dp, sV, tdO, warp, lane);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int qc = nt * 8 + (lane & 3) * 2;
            const float e0 = tD[qc], e1 = tD[qc + 1];
            s[nt][0] *= (dp[nt][0] - e0) * p.scale;
            s[nt][1] *= (dp[nt][1] - e1) * p.scale;
            s[nt][2] *= (dp[nt][2] - e0) * p.scale;
            s[nt][3] *= (dp[nt][3] - e1) * p.scale;
        }
        // dK += dS^T Q
        mma_acc_x_rows<NKS, PITCH>(dk, s, tQ, d0, lane);
    }
    const int r0 = k0 + warp * 16 + (lane >> 2), r1 = r0 + 8;
#pragma unroll
    for (int nt = 0; nt < 2 * NKS; ++nt) {
        const int col = d0 + nt * 8 + (lane & 3) * 2;
        if (col < D) {
            if (r0 < p.Skv) {
                *reinterpret_cast<uint32_t*>(p.dk + ((size_t)b * p.Skv + r0) * p.lddk + h * D + col) = pack_bf16x2(dk[nt][0], dk[nt][1]);
                *reinterpret_cast<uint32_t*>(p.dv + ((size_t)b * p.Skv + r0) * p.lddv + h * D + col) = pack_bf16x2(dv[nt][0], dv[nt][1]);
            }
            if (r1 < p.Skv) {
                *reinterpret_cast<uint32_t*>(p.dk + ((size_t)b * p.Skv + r1) * p.lddk + h * D + col) = pack_bf16x2(dk[nt][2], dk[nt][3]);
                *reinterpret_cast<uint32_t*>(p.dv + ((size_t)b * p.Skv + r1) * p.lddv + h * D + col) = pack_bf16x2(dv[nt][2], dv[nt][3]);
            }
        }
    }
}

template <int DP>
int launch_bwd(const BwdParams& p, int batch, cudaStream_t s) {
    constexpr int PITCH = DP * 2 + 16;
    constexpr int DSPLIT = (DP > 96 && (DP / 16) % 2 == 0) ? 2 : 1;
    const size_t smem_dq = (size_t)6 * kT * PITCH;
    const size_t smem_dkv = (size_t)6 * kT * PITCH + 4 * kT * sizeof(float);
    B200SD_CUDA(b200sd_opt_in_smem(attn_bwd_dq_kernel<DP>, (int)smem_dq));
    B200SD_CUDA(b200sd_opt_in_smem(attn_bwd_dkv_kernel<DP, DSPLIT>, (int)smem_dkv));
    attn_bwd_dq_kernel<DP><<<dim3(ceil_div(p.Sq, kT), p.heads, batch), dim3(kThreads), smem_dq, s>>>(p);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    attn_bwd_dkv_kernel<DP, DSPLIT><<<dim3(ceil_div(p.Skv, kT) * DSPLIT, p.heads, batch), dim3(kThreads), smem_dkv, s>>>(p);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

}  // namespace

int b200sd_attention_bwd_tc(const bf16* q, const bf16* k, const bf16* v, const bf16* dout, const float* lse, const float* delta,
                            bf16* dq, bf16* dk, bf16* dv, int batch, int heads, int Sq, int Skv, int d, int ldq, int ldk,
                            int ldv, int lddo, int lddq, int lddk, int lddv, float scale, cudaStream_t s);

extern "C" size_t b200sd_attention_bwd_workspace_bytes(int batch, int heads, int Sq) {
    return (size_t)batch * heads * Sq * sizeof(float);
}

extern "C" int b200sd_attention_bwd(const void* q, const void* k, const void* v, const void* out, const void* dout,
                                    const float* lse, void* dq, void* dk, void* dv, int batch, int heads, int Sq, int Skv,
                                    int d, int ldq, int ldk, int ldv, int ldo, int lddo, int lddq, int lddk, int lddv,
                                    float scale, void* workspace, size_t workspace_bytes, b200sd_stream_t stream) {
    B200SD_REQUIRE(q && k && v && out && dout && lse && dq && dk && dv && workspace, "attention_bwd: null pointer");
    B200SD_REQUIRE(batch > 0 && heads > 0 && Sq > 0 && Skv > 0 && batch <= 65535 && heads <= 65535, "attention_bwd: bad sizes");
    B200SD_REQUIRE(d % 8 == 0 && d >= 8 && d <= 160, "attention_bwd: head dim %d unsupported (multiple of 8, <= 160)", d);
    B200SD_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0 && lddo % 8 == 0 && lddq % 2 == 0 && lddk % 2 == 0 && lddv % 2 == 0,
                   "attention_bwd: leading dims must be multiples of 8");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                     reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(dout)) & 15) == 0 &&
                       ((reinterpret_cast<uintptr_t>(dq) | reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv)) & 3) == 0,
                   "attention_bwd: pointers must be 16-byte aligned");
    B200SD_REQUIRE(workspace_bytes >= b200sd_attention_bwd_workspace_bytes(batch, heads, Sq), "attention_bwd: workspace too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float* delta = static_cast<float*>(workspace);
    {
        const int64_t total = (int64_t)batch * Sq * heads;
        int blocks = (int)((total + 255) / 256);
        const int cap = b200sd_num_sms() * 8;
        if (blocks > cap) blocks = cap;
        attn_delta_kernel<<<dim3(blocks), dim3(256), 0, s>>>(static_cast<const bf16*>(out), static_cast<const bf16*>(dout),
                                  delta, batch, heads, Sq, d, ldo, lddo);
        COUNT_LAUNCH();
        B200SD_LAUNCH_CHECK();
    }
    {
        // tensor-core (tcgen05 / TMEM) kernels for the self-attention-sized shapes
        const int rc = b200sd_attention_bwd_tc(static_cast<const bf16*>(q), static_cast<const bf16*>(k), static_cast<const bf16*>(v),
                                               static_cast<const bf16*>(dout), lse, delta, static_cast<bf16*>(dq), static_cast<bf16*>(dk),
                                               static_cast<bf16*>(dv), batch, heads, Sq, Skv, d, ldq, ldk, ldv, lddo, lddq, lddk, lddv,
                                               scale, s);
        if (rc != B200SD_ERR_UNSUPPORTED) return rc;
    }
    BwdParams p;
    p.q = static_cast<const bf16*>(q); p.k = static_cast<const bf16*>(k); p.v = static_cast<const bf16*>(v);
    p.dout = static_cast<const bf16*>(dout);
    p.lse = lse; p.delta = delta;
    p.dq = static_cast<bf16*>(dq); p.dk = static_cast<bf16*>(dk); p.dv = static_cast<bf16*>(dv);
    p.Sq = Sq; p.Skv = Skv; p.D = d; p.heads = heads;
    p.ldq = ldq; p.ldk = ldk; p.ldv = ldv; p.ldo = lddo; p.lddq = lddq; p.lddk = lddk; p.lddv = lddv;
    p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
    const int dp = (d + 15) / 16 * 16;
#define BWD_CASE(DP) case DP: return launch_bwd<DP>(p, batch, s);
    switch (dp) {
        BWD_CASE(16) BWD_CASE(32) BWD_CASE(48) BWD_CASE(64) BWD_CASE(80) BWD_CASE(96) BWD_CASE(112) BWD_CASE(128)
        BWD_CASE(144) BWD_CASE(160)
    }
#undef BWD_CASE
    B200SD_REQUIRE(false, "attention_bwd: head dim %d unsupported", d);
}
