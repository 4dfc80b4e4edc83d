// b200sd -- fused (flash-style) attention: out = softmax(scale * Q K^T) V, never materialising the
// S x S score matrix (the reference's baddbmm + softmax + bmm, SURVEY.md K4).
//
// Round-1 implementation: register-resident online softmax with warp-level tensor-core MMA
// (mma.sync m16n8k16 bf16, fp32 accumulate), cp.async double-buffered K/V tiles, 128 query rows per
// CTA (8 warps x 16 rows), 64 keys per tile.  Head dims 40/80/160 are padded to a multiple of 16 in
// shared memory (zero-filled), key tails (S_kv = 77) are masked to -inf.  The tcgen05/TMEM version
// of this kernel is the next step for this row (DESIGN.md).
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;

namespace {

constexpr int kBM = 128;  // query rows per CTA
constexpr int kBN = 64;   // keys per tile
constexpr int kThreads = 256;

__device__ __forceinline__ void cp_async16(void* dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ptx::smem_u32(dst)), "l"(src), "r"(src_bytes)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(ptx::smem_u32(p)));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(ptx::smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
        "{%0, %1, %2, %3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows x (D/8) 16-byte chunks, global [row][ld] -> smem [row][PITCH]; rows beyond `valid` zero-filled
template <int PITCH>
__device__ __forceinline__ void load_tile(uint8_t* smem, const bf16* g, int ld, int rows, int valid, int chunks) {
    for (int i = threadIdx.x; i < rows * chunks; i += kThreads) {
        const int r = i / chunks, c = i % chunks;
        const bool ok = r < valid;
        const bf16* src = g + (size_t)(ok ? r : 0) * ld + c * 8;
        cp_async16(smem + (size_t)r * PITCH + c * 16, src, ok ? 16 : 0);
    }
}

template <int DP>
__global__ void __launch_bounds__(kThreads, (DP <= 80) ? 2 : 1)
    attention_kernel(const bf16* __restrict__ q, const bf16* __restrict__ k, const bf16* __restrict__ v,
                     bf16* __restrict__ out, float* __restrict__ lse, int Sq, int Skv, int D, int ldq, int ldk, int ldv,
                     int ldo, float scale_log2) {
    constexpr int PITCH = DP * 2 + 16;
    constexpr int KS = DP / 16;  // k-steps over the head dim
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* sQ = smem;
    uint8_t* sK = sQ + kBM * PITCH;
    uint8_t* sV = sK + 2 * kBN * PITCH;

    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * kBM;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunks = D / 8;

    // zero the head-dim padding once (cp.async never touches it)
    {
        constexpr int PAD16 = PITCH / 16;  // 16-byte slots per row incl. the bank-skew slot
        const int total_rows = kBM + 4 * kBN;
        for (int i = threadIdx.x; i < total_rows * (PAD16 - chunks); i += kThreads) {
            const int r = i / (PAD16 - chunks), c = chunks + i % (PAD16 - chunks);
            *reinterpret_cast<uint4*>(smem + (size_t)r * PITCH + c * 16) = make_uint4(0, 0, 0, 0);
        }
    }

    const bf16* qg = q + ((size_t)b * Sq + q0) * ldq + h * D;
    const bf16* kg = k + (size_t)b * Skv * ldk + h * D;
    const bf16* vg = v + (size_t)b * Skv * ldv + h * D;
    const int num_tiles = (Skv + kBN - 1) / kBN;

    load_tile<PITCH>(sQ, qg, ldq, kBM, min(kBM, Sq - q0), chunks);
    load_tile<PITCH>(sK, kg, ldk, kBN, min(kBN, Skv), chunks);
    load_tile<PITCH>(sV, vg, ldv, kBN, min(kBN, Skv), chunks);
    cp_async_commit();

    uint32_t qf[KS][4];
    float o[2 * KS][4];
#pragma unroll
    for (int i = 0; i < 2 * KS; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    for (int j = 0; j < num_tiles; ++j) {
        cp_async_wait<0>();
        __syncthreads();
        if (j == 0) {
#pragma unroll
            for (int ks = 0; ks < KS; ++ks)
                ldmatrix_x4(qf[ks], sQ + (size_t)(warp * 16 + (lane & 15)) * PITCH + (ks * 16 + (lane >> 4) * 8) * 2);
        }
        if (j + 1 < num_tiles) {
            const int nb = (j + 1) & 1;
            const int valid = min(kBN, Skv - (j + 1) * kBN);
            load_tile<PITCH>(sK + (size_t)nb * kBN * PITCH, kg + (size_t)(j + 1) * kBN * ldk, ldk, kBN, valid, chunks);
            load_tile<PITCH>(sV + (size_t)nb * kBN * PITCH, vg + (size_t)(j + 1) * kBN * ldv, ldv, kBN, valid, chunks);
            cp_async_commit();
        }
        const uint8_t* tK = sK + (size_t)(j & 1) * kBN * PITCH;
        const uint8_t* tV = sV + (size_t)(j & 1) * kBN * PITCH;

        // ---- S = Q K^T (16 x 64 per warp) ----
        float s[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
                uint32_t kf[4];
                ldmatrix_x4(kf, tK + (size_t)(np * 16 + (lane & 7) + (lane >> 4) * 8) * PITCH +
                                    (ks * 16 + ((lane >> 3) & 1) * 8) * 2);
                mma_bf16(s[2 * np], qf[ks], kf[0], kf[1]);
                mma_bf16(s[2 * np + 1], qf[ks], kf[2], kf[3]);
            }
        }
        // ---- mask the key tail ----
        const int kbase = j * kBN;
        if (kbase + kBN > Skv) {
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int key = kbase + nt * 8 + (lane & 3) * 2;
                if (key >= Skv) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
                if (key + 1 >= Skv) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
            }
        }
        // ---- online softmax ----
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
            mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
        const float corr0 = exp2f((m0 - mn0) * scale_log2), corr1 = exp2f((m1 - mn1) * scale_log2);
        const float off0 = mn0 * scale_log2, off1 = mn1 * scale_log2;
        m0 = mn0;
        m1 = mn1;
        float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            s[nt][0] = exp2f(s[nt][0] * scale_log2 - off0);
            s[nt][1] = exp2f(s[nt][1] * scale_log2 - off0);
            s[nt][2] = exp2f(s[nt][2] * scale_log2 - off1);
            s[nt][3] = exp2f(s[nt][3] * scale_log2 - off1);
            rs0 += s[nt][0] + s[nt][1];
            rs1 += s[nt][2] + s[nt][3];
        }
        l0 = l0 * corr0 + rs0;
        l1 = l1 * corr1 + rs1;
#pragma unroll
        for (int i = 0; i < 2 * KS; ++i) {
            o[i][0] *= corr0; o[i][1] *= corr0;
            o[i][2] *= corr1; o[i][3] *= corr1;
        }
        // ---- O += P V ----
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t a[4];
            a[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
            a[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
            a[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
            a[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
            for (int dp = 0; dp < KS; ++dp) {
                uint32_t vf[4];
                ldmatrix_x4_trans(vf, tV + (size_t)(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * PITCH +
                                          (dp * 16 + (lane >> 4) * 8) * 2);
                mma_bf16(o[2 * dp], a, vf[0], vf[1]);
                mma_bf16(o[2 * dp + 1], a, vf[2], vf[3]);
            }
        }
    }

    // ---- finalize ----
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
    const int r0 = q0 + warp * 16 + (lane >> 2), r1 = r0 + 8;
    if (lse != nullptr && (lane & 3) == 0) {   // log2-domain log-sum-exp of the scaled scores (saved for the backward)
        float* dst = lse + ((size_t)b * gridDim.y + h) * Sq;
        if (r0 < Sq) dst[r0] = m0 * scale_log2 + log2f(l0);
        if (r1 < Sq) dst[r1] = m1 * scale_log2 + log2f(l1);
    }
#pragma unroll
    for (int nt = 0; nt < 2 * KS; ++nt) {
        const int col = nt * 8 + (lane & 3) * 2;
        if (col < D) {
            if (r0 < Sq)
                *reinterpret_cast<uint32_t*>(out + ((size_t)b * Sq + r0) * ldo + h * D + col) =
                    pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
            if (r1 < Sq)
                *reinterpret_cast<uint32_t*>(out + ((size_t)b * Sq + r1) * ldo + h * D + col) =
                    pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
        }
    }
}

template <int DP>
int launch_attention(const bf16* q, const bf16* k, const bf16* v, bf16* out, float* lse, int batch, int heads, int Sq, int Skv,
                     int D, int ldq, int ldk, int ldv, int ldo, float scale, cudaStream_t s) {
    constexpr int PITCH = DP * 2 + 16;
    const size_t smem = (size_t)(kBM + 4 * kBN) * PITCH;
    B200SD_CUDA(b200sd_opt_in_smem(attention_kernel<DP>, (int)smem));
    dim3 grid(ceil_div(Sq, kBM), heads, batch);
    attention_kernel<DP><<<dim3(grid), dim3(kThreads), smem, s>>>(q, k, v, out, lse, Sq, Skv, D, ldq, ldk, ldv, ldo,
                                                      scale * 1.4426950408889634f);
    g_b200sd_launches.fetch_add(1, std::memory_order_relaxed);
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

}  // namespace

int b200sd_attention_tc(const void* q, const void* k, const void* v, void* out, float* lse, int batch, int heads, int Sq, int Skv,
                        int d, int ldq, int ldk, int ldv, int ldo, float scale, void* workspace, size_t ws_bytes,
                        cudaStream_t s);

// The tcgen05 kernel used to need a V^T scratch copy; it now reads V in place, so no workspace is required any more.
// The entry point stays in the ABI (callers size their buffer with it) and returns 0.
extern "C" size_t b200sd_attention_workspace_bytes(int batch, int heads, int Skv, int d) {
    (void)batch; (void)heads; (void)Skv; (void)d;
    return 0;
}

extern "C" int b200sd_attention_lse(const void* q, const void* k, const void* v, void* out, float* lse, int batch, int heads,
                                    int Sq, int Skv, int d, int ldq, int ldk, int ldv, int ldo, float scale,
                                    void* workspace, size_t workspace_bytes, b200sd_stream_t stream) {
    B200SD_REQUIRE(q && k && v && out, "attention: null pointer");
    B200SD_REQUIRE(batch > 0 && heads > 0 && Sq > 0 && Skv > 0, "attention: bad sizes");
    B200SD_REQUIRE(batch <= 65535 && heads <= 65535, "attention: batch/heads too large");
    B200SD_REQUIRE(d % 8 == 0 && d >= 8 && d <= 160, "attention: head dim %d unsupported (multiple of 8, <= 160)", d);
    B200SD_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 2 == 0, "attention: leading dims must be multiples of 8");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(out) & 3) == 0,
                   "attention: pointers must be 16-byte aligned");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    {
        // tensor-core (tcgen05/TMEM) path for the self-attention-sized shapes
        const int rc = b200sd_attention_tc(q, k, v, out, lse, batch, heads, Sq, Skv, d, ldq, ldk, ldv, ldo, scale, workspace,
                                           workspace_bytes, s);
        if (rc != B200SD_ERR_UNSUPPORTED) return rc;
    }
    const bf16* qq = static_cast<const bf16*>(q);
    const bf16* kk = static_cast<const bf16*>(k);
    const bf16* vv = static_cast<const bf16*>(v);
    bf16* oo = static_cast<bf16*>(out);
    const int dp = (d + 15) / 16 * 16;
#define ATT_CASE(DP) \
    case DP: return launch_attention<DP>(qq, kk, vv, oo, lse, batch, heads, Sq, Skv, d, ldq, ldk, ldv, ldo, scale, s);
    switch (dp) {
        ATT_CASE(16) ATT_CASE(32) ATT_CASE(48) ATT_CASE(64) ATT_CASE(80) ATT_CASE(96) ATT_CASE(112) ATT_CASE(128)
        ATT_CASE(144) ATT_CASE(160)
    }
#undef ATT_CASE
    B200SD_REQUIRE(false, "attention: head dim %d unsupported", d);
}

extern "C" int b200sd_attention(const void* q, const void* k, const void* v, void* out, int batch, int heads, int Sq,
                                int Skv, int d, int ldq, int ldk, int ldv, int ldo, float scale,
                                void* workspace, size_t workspace_bytes, b200sd_stream_t stream) {
    return b200sd_attention_lse(q, k, v, out, nullptr, batch, heads, Sq, Skv, d, ldq, ldk, ldv, ldo, scale, workspace,
                                workspace_bytes, stream);
}
