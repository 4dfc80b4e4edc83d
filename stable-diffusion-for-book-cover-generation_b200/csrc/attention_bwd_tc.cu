// b200sd -- flash-attention BACKWARD on the sm_100a tensor cores (tcgen05 + TMEM), self-attention sized: head dim 40 / 80,
// S_q and S_kv multiples of 128 (the 64x64 and 32x32 levels: 98 % of the attention-backward FLOPs).  Other shapes keep
// the mma.sync kernels in attention_bwd.cu.
//
// One templated kernel, two roles (both deterministic, no atomics):
//   DKV : CTA owns 128 keys (K, V stationary in smem), streams 128-query tiles (Q, dO, lse, delta):
//           S^T = K Q^T, dP^T = V dO^T  (TMEM)  ->  P^T = exp2(S^T sl2 - lse[q]),  dS^T = P^T (dP^T - delta[q])
//           dV += P^T dO,  dK += dS^T Q          (accumulators stay in TMEM for the whole key tile)
//   DQ  : CTA owns 128 queries (Q, dO stationary), streams 128-key tiles (K, V):
//           S = Q K^T, dP = dO V^T  ->  dS = exp2(S sl2 - lse[row]) (dP - delta[row]);  dQ += dS K
// Every operand is consumed in its natural [row][d] layout: the first two products read both operands K-major, the
// accumulating products read the streamed tile as an MN-major B operand (UMMA transpose descriptor over the same
// SWIZZLE_128B TMA box), so no transposed copy of anything exists.  The q/k/v/dO buffers are addressed as 3-D tensors
// (d, head, row): a 64-wide box over a 40-wide head is zero-filled past the head by TMA.
//   warp 0    : TMA producer;  warp 1 : TMEM allocator + single-thread MMA issuer
//   warps 2-9 : 256 compute threads: thread = one accumulator row (TMEM lane) x one 64-column half of the tile;
//               tcgen05.ld, exp2 / FMA in fp32, bf16 P^T / dS^T written into 128B-swizzled smem tiles (the A operands
//               of the accumulating MMAs); at the end the accumulators are scaled and stored as bf16.
#include <atomic>
#include <cstring>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;

namespace {

constexpr int kT = 128;                 // tile edge (stationary rows and streamed rows)
constexpr int kThreads = 320;           // producer warp + MMA warp + 8 compute warps
constexpr int kBlk = kT * 128;          // bytes of one [128 rows x 64 bf16] swizzled block

struct BwdTcParams {
    CUtensorMap tmX1, tmX2, tmY1, tmY2;   // stationary (K, V | Q, dO) and streamed (Q, dO | K, V) operands
    const float* lse;                     // [batch][heads][Sq], log2 domain
    const float* delta;                   // [batch][heads][Sq]
    bf16* out1;                           // DKV: dV;  DQ: unused
    bf16* out2;                           // DKV: dK;  DQ: dQ
    int Sx, Sy, heads, ld1, ld2;          // rows of the stationary / streamed sequence; leading dims of out1 / out2
    float scale, scale_log2;
};

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// packed fp32x2 math (FFMA2 / FADD2 / FMUL2): halves the non-MUFU instructions of the compute warps
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ptx::smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(ptx::smem_u32(bar))
                 : "memory");
}

// D = head dim (40 / 80); DKB = 64-wide blocks covering it; STAGES = ring depth of the streamed operands
// ATMEM: P^T / dS^T (the A operands of the accumulating products) are handed to the tensor core through TMEM
// (tcgen05.st by the compute threads, tcgen05.mma with the A operand in TMEM) instead of 64 KB of swizzled smem tiles:
// the kernel is shared-memory-bandwidth bound otherwise (~256 KB of smem traffic per 128x128 tile pair).
template <int D, int DKB, int STAGES, bool DKV, bool ATMEM>
__global__ void __launch_bounds__(kThreads, 1) attn_bwd_tc_kernel(const __grid_constant__ BwdTcParams p) {
    constexpr int DN = (D + 15) / 16 * 16;     // MMA N of the accumulating products (48 / 80)
    constexpr int KSTEPS = (D + 15) / 16;      // UMMA K steps over the head dim
    constexpr uint32_t kTmemCols = 512;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sX1 = smem;                                  // DKB blocks
    uint8_t* sX2 = sX1 + DKB * kBlk;
    uint8_t* sY1 = sX2 + DKB * kBlk;                      // STAGES x DKB blocks
    uint8_t* sY2 = sY1 + STAGES * DKB * kBlk;
    uint8_t* sP = sY2 + STAGES * DKB * kBlk;              // 2 blocks (DKV only, but always reserved)
    uint8_t* sdS = sP + 2 * kBlk;                         // 2 blocks
    float* sVec = reinterpret_cast<float*>(sdS + 2 * kBlk);   // [STAGES][2][128]: lse, delta of the streamed queries (DKV)
    uint64_t* bars = reinterpret_cast<uint64_t*>(sVec + STAGES * 2 * kT);
    uint64_t* x_full = bars;
    uint64_t* y_full = bars + 1;              // [STAGES]
    uint64_t* y_empty = bars + 1 + STAGES;    // [STAGES]
    uint64_t* t_full = bars + 1 + 2 * STAGES;   // [2]: one per 64-row half of the streamed tile
    uint64_t* p_full = t_full + 2;              // [2]
    uint64_t* p_empty = t_full + 4;             // [2]
    uint64_t* acc_full = t_full + 6;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_full + 7);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int x0 = blockIdx.x * kT, h = blockIdx.y, b = blockIdx.z;
    const int num_tiles = p.Sy / kT;
    const int Sq = DKV ? p.Sy : p.Sx;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&p.tmX1);
        ptx::prefetch_tmap(&p.tmX2);
        ptx::prefetch_tmap(&p.tmY1);
        ptx::prefetch_tmap(&p.tmY2);
        ptx::mbar_init(x_full, 1);
        for (int i = 0; i < STAGES; ++i) {
            ptx::mbar_init(&y_full[i], 1);
            ptx::mbar_init(&y_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&t_full[i], 1);
            ptx::mbar_init(&p_full[i], 256);
            ptx::mbar_init(&p_empty[i], 1);
        }
        ptx::mbar_init(acc_full, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc(tmem_slot, kTmemCols);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // TMEM columns: T1 [0,128) T2 [128,256); accumulators A1 [256,..) A2 [320,..) (ATMEM) or [384,..);
    // ATMEM: P^T operand [384,448), dS^T operand [448,512): 64 bf16 (= 32 columns) per 64-row half of the streamed tile
    const uint32_t tT1 = tmem_base, tT2 = tmem_base + 128, tA1 = tmem_base + 256, tA2 = tmem_base + (ATMEM ? 320 : 384);
    const uint32_t tP = tmem_base + 384, tdS = tmem_base + 448;

    if (warp == 0) {
        // ================= TMA producer =================
        if (ptx::elect_one()) {
            ptx::mbar_expect_tx(x_full, 2 * DKB * kBlk);
            for (int kb = 0; kb < DKB; ++kb) {
                ptx::tma_load_3d(sX1 + kb * kBlk, &p.tmX1, x_full, kb * 64, h, b * p.Sx + x0);
                ptx::tma_load_3d(sX2 + kb * kBlk, &p.tmX2, x_full, kb * 64, h, b * p.Sx + x0);
            }
            const size_t vec_base = ((size_t)b * p.heads + h) * Sq;
            for (int j = 0; j < num_tiles; ++j) {
                const int st = j % STAGES;
                const uint32_t ph = (uint32_t)(j / STAGES) & 1;
                ptx::mbar_wait(&y_empty[st], ph ^ 1);
                ptx::mbar_expect_tx(&y_full[st], 2 * DKB * kBlk + (DKV ? 2 * kT * 4 : 0));
                for (int kb = 0; kb < DKB; ++kb) {
                    ptx::tma_load_3d(sY1 + (st * DKB + kb) * kBlk, &p.tmY1, &y_full[st], kb * 64, h, b * p.Sy + j * kT);
                    ptx::tma_load_3d(sY2 + (st * DKB + kb) * kBlk, &p.tmY2, &y_full[st], kb * 64, h, b * p.Sy + j * kT);
                }
                if constexpr (DKV) {
                    bulk_load_1d(sVec + (st * 2) * kT, p.lse + vec_base + (size_t)j * kT, kT * 4, &y_full[st]);
                    bulk_load_1d(sVec + (st * 2 + 1) * kT, p.delta + vec_base + (size_t)j * kT, kT * 4, &y_full[st]);
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        // Software-pipelined over the two 64-row halves of every streamed tile: while the compute warps work on one half the
        // tensor core runs the products of the other, and the next tile's first products are issued as soon as its TMEM
        // columns have been read.
        if (ptx::elect_one()) {
            const uint32_t idesc_t = ptx::umma_idesc_bf16(128, 64);
            const uint32_t idesc_a = ptx::umma_idesc_bf16(128, DN) | (1u << 16);   // B operand MN-major
            auto issue_T = [&](int st, int half) {   // T1 / T2 columns [half*64, +64): X (128 rows) x 64 streamed rows, K over d
#pragma unroll
                for (int ks = 0; ks < KSTEPS; ++ks) {
                    const int kb = ks / 4, kin = ks % 4;
                    const uint64_t da = ptx::umma_desc_k_sw128(ptx::smem_u32(sX1 + kb * kBlk)) + 2 * kin;
                    const uint64_t db = ptx::umma_desc_k_sw128(ptx::smem_u32(sY1 + (st * DKB + kb) * kBlk) + half * 8192) + 2 * kin;
                    ptx::umma_bf16_ss(tT1 + half * 64, da, db, idesc_t, ks > 0 ? 1u : 0u);
                }
#pragma unroll
                for (int ks = 0; ks < KSTEPS; ++ks) {
                    const int kb = ks / 4, kin = ks % 4;
                    const uint64_t da = ptx::umma_desc_k_sw128(ptx::smem_u32(sX2 + kb * kBlk)) + 2 * kin;
                    const uint64_t db = ptx::umma_desc_k_sw128(ptx::smem_u32(sY2 + (st * DKB + kb) * kBlk) + half * 8192) + 2 * kin;
                    ptx::umma_bf16_ss(tT2 + half * 64, da, db, idesc_t, ks > 0 ? 1u : 0u);
                }
                ptx::umma_commit(&t_full[half]);
            };
            auto issue_acc = [&](int j, int st, int half) {   // A2 += dS Y1 (A1 += P Y2): 64 streamed rows = 4 k-steps
#pragma unroll
                for (int kin = 0; kin < 4; ++kin) {
                    const int ks = half * 4 + kin;
                    const uint32_t acc = (j > 0 || ks > 0) ? 1u : 0u;
                    if constexpr (DKV) {
                        const uint64_t db = ptx::umma_desc_mn_sw128(ptx::smem_u32(sY2 + st * DKB * kBlk) + ks * 2048, kBlk);
                        if constexpr (ATMEM) ptx::umma_bf16_ts(tA1, tP + half * 32 + kin * 8, db, idesc_a, acc);
                        else ptx::umma_bf16_ss(tA1, ptx::umma_desc_k_sw128(ptx::smem_u32(sP + half * kBlk)) + 2 * kin, db, idesc_a, acc);
                    }
                    const uint64_t db2 = ptx::umma_desc_mn_sw128(ptx::smem_u32(sY1 + st * DKB * kBlk) + ks * 2048, kBlk);
                    if constexpr (ATMEM) ptx::umma_bf16_ts(tA2, tdS + half * 32 + kin * 8, db2, idesc_a, acc);
                    else ptx::umma_bf16_ss(tA2, ptx::umma_desc_k_sw128(ptx::smem_u32(sdS + half * kBlk)) + 2 * kin, db2, idesc_a, acc);
                }
                ptx::umma_commit(&p_empty[half]);
            };
            ptx::mbar_wait(x_full, 0);
            ptx::mbar_wait(&y_full[0], 0);
            ptx::tc_fence_after();
            issue_T(0, 0);
            issue_T(0, 1);
            for (int j = 0; j < num_tiles; ++j) {
                const int st = j % STAGES, stn = (j + 1) % STAGES;
                const bool more = j + 1 < num_tiles;
                ptx::mbar_wait(&p_full[0], j & 1);           // half 0 of tile j: T columns read, P / dS written
                ptx::tc_fence_after();
                issue_acc(j, st, 0);
                if (more && STAGES > 1) {
                    ptx::mbar_wait(&y_full[stn], (uint32_t)((j + 1) / STAGES) & 1);
                    ptx::tc_fence_after();
                    issue_T(stn, 0);
                }
                ptx::mbar_wait(&p_full[1], j & 1);
                ptx::tc_fence_after();
                issue_acc(j, st, 1);
                ptx::umma_commit(&y_empty[st]);
                if (more) {
                    if (STAGES == 1) {   // single-stage ring: the next tile can only land after this one has been consumed
                        ptx::mbar_wait(&y_full[stn], (uint32_t)((j + 1) / STAGES) & 1);
                        ptx::tc_fence_after();
                        issue_T(stn, 0);
                    }
                    issue_T(stn, 1);
                }
            }
            ptx::umma_commit(acc_full);
        }
    } else {
        // ================= compute warps: thread = accumulator row x 64-column half =================
        const int qd = warp & 3, half = (warp - 2) >> 2;
        const int row = qd * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(qd * 32) << 16;
        float lse_r = 0.f, del_r = 0.f;
        if constexpr (!DKV) {
            const size_t vb = ((size_t)b * p.heads + h) * Sq + x0 + row;
            lse_r = p.lse[vb];
            del_r = p.delta[vb];
        }
        for (int j = 0; j < num_tiles; ++j) {
            const int st = j % STAGES;
            const float* lse_s = sVec + (st * 2) * kT;
            const float* del_s = sVec + (st * 2 + 1) * kT;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {             // the two 64-row halves of the streamed tile
                ptx::mbar_wait(&t_full[hh], j & 1);
                ptx::tc_fence_after();
                if (j > 0) ptx::mbar_wait(&p_empty[hh], (j - 1) & 1);   // the previous tile's accumulating MMAs have read this block
                const int cc = half * 32;                // this thread's 32 columns inside the 64-column half
                const int c = hh * 64 + cc;
                uint32_t r1[32], r2[32];
                tmem_ld_x32(tT1 + lane_addr + c, r1);
                tmem_ld_x32(tT2 + lane_addr + c, r2);
                ptx::tmem_ld_wait();
                uint32_t pk[16], dk[16];
#pragma unroll
                const float2 sl2v = make_float2(p.scale_log2, p.scale_log2);
                for (int i = 0; i < 16; ++i) {
                    float2 nl, dl;     // -lse and delta of this column pair
                    if constexpr (DKV) {
                        const float2 lv = *reinterpret_cast<const float2*>(lse_s + c + 2 * i);
                        nl = make_float2(-lv.x, -lv.y);
                        dl = *reinterpret_cast<const float2*>(del_s + c + 2 * i);
                    } else {
                        nl = make_float2(-lse_r, -lse_r);
                        dl = make_float2(del_r, del_r);
                    }
                    const float2 t = ffma2(make_float2(__uint_as_float(r1[2 * i]), __uint_as_float(r1[2 * i + 1])), sl2v, nl);
                    const float2 pe = make_float2(fast_exp2(t.x), fast_exp2(t.y));
                    const float2 ds = fmul2(pe, fsub2(make_float2(__uint_as_float(r2[2 * i]), __uint_as_float(r2[2 * i + 1])), dl));
                    pk[i] = pack_bf16x2(pe.x, pe.y);
                    dk[i] = pack_bf16x2(ds.x, ds.y);
                }
                if constexpr (ATMEM) {
                    // this thread's 32 streamed rows = 16 packed columns of its lane in the A-operand region of this half
                    if constexpr (DKV) tmem_st_x16(tP + lane_addr + hh * 32 + half * 16, pk);
                    tmem_st_x16(tdS + lane_addr + hh * 32 + half * 16, dk);
                    ptx::tmem_st_wait();
                    ptx::tc_fence_before();
                } else {
                    uint8_t* bp = sP + hh * kBlk + row * 128;
                    uint8_t* bd = sdS + hh * kBlk + row * 128;
#pragma unroll
                    for (int g = 0; g < 4; ++g) {   // four 16-byte chunks (8 streamed rows each) of this 32-column piece
                        const int chunk = (cc / 8 + g) ^ (row & 7);
                        if constexpr (DKV) *reinterpret_cast<uint4*>(bp + chunk * 16) = make_uint4(pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
                        *reinterpret_cast<uint4*>(bd + chunk * 16) = make_uint4(dk[4 * g], dk[4 * g + 1], dk[4 * g + 2], dk[4 * g + 3]);
                    }
                    ptx::tc_fence_before();
                    ptx::fence_proxy_async();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
                }
                ptx::mbar_arrive(&p_full[hh]);
            }
        }
        // ---- accumulators -> bf16 global (row per thread; half 0 stores A1 = dV, half 1 stores A2 = dK / dQ (scaled)) ----
        ptx::mbar_wait(acc_full, 0);
        ptx::tc_fence_after();
        if (DKV || half == 1) {
            const uint32_t tacc = (half == 0 ? tA1 : tA2) + lane_addr;
            const float mul = half == 0 ? 1.0f : p.scale;
            bf16* base = half == 0 ? p.out1 : p.out2;
            const int ld = half == 0 ? p.ld1 : p.ld2;
            bf16* dst = base + ((size_t)b * p.Sx + x0 + row) * ld + h * D;
#pragma unroll
            for (int c = 0; c < DN; c += 16) {
                uint32_t r[16];
                ptx::tmem_ld_32x32b_x16(tacc + c, r);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    if (c + 8 * g < D) {
                        uint4 u;
                        u.x = pack_bf16x2(__uint_as_float(r[8 * g]) * mul, __uint_as_float(r[8 * g + 1]) * mul);
                        u.y = pack_bf16x2(__uint_as_float(r[8 * g + 2]) * mul, __uint_as_float(r[8 * g + 3]) * mul);
                        u.z = pack_bf16x2(__uint_as_float(r[8 * g + 4]) * mul, __uint_as_float(r[8 * g + 5]) * mul);
                        u.w = pack_bf16x2(__uint_as_float(r[8 * g + 6]) * mul, __uint_as_float(r[8 * g + 7]) * mul);
                        *reinterpret_cast<uint4*>(dst + c + 8 * g) = u;
                    }
                }
            }
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, kTmemCols);
    }
}

int make_map(CUtensorMap* m, const bf16* ptr, int D, int heads, int64_t rows, int ld) {
    const uint64_t dims[3] = {(uint64_t)D, (uint64_t)heads, (uint64_t)rows};
    const uint64_t str[3] = {0, (uint64_t)D * 2, (uint64_t)ld * 2};
    const uint32_t box[3] = {64, 1, 128};
    return b200sd_make_tmap(m, ptr, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int D, int DKB, int STAGES, bool DKV, bool ATMEM>
int launch_one(const BwdTcParams& p, int batch, cudaStream_t s) {
    const size_t smem = (size_t)(2 * DKB + 2 * STAGES * DKB + 4) * kBlk + STAGES * 2 * kT * 4 + 256 + 1024;
    B200SD_CUDA(b200sd_opt_in_smem(attn_bwd_tc_kernel<D, DKB, STAGES, DKV, ATMEM>, (int)smem));
    attn_bwd_tc_kernel<D, DKB, STAGES, DKV, ATMEM><<<dim3(p.Sx / kT, p.heads, batch), dim3(kThreads), smem, s>>>(p);
    g_b200sd_launches.fetch_add(1, std::memory_order_relaxed);
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

}  // namespace

// Returns B200SD_ERR_UNSUPPORTED when the shape is not covered (the caller falls back to the mma.sync kernels).
// delta must already hold rowsum(dO o O).
int b200sd_attention_bwd_tc(const bf16* q, const bf16* k, const bf16* v, const bf16* dout, const float* lse, const float* delta,
                            bf16* dq, bf16* dk, bf16* dv, int batch, int heads, int Sq, int Skv, int d, int ldq, int ldk,
                            int ldv, int lddo, int lddq, int lddk, int lddv, float scale, cudaStream_t s) {
    if (!(d == 40 || d == 80) || Sq % kT != 0 || Skv % kT != 0) return B200SD_ERR_UNSUPPORTED;
    if ((ldq * 2) % 16 != 0 || (ldk * 2) % 16 != 0 || (ldv * 2) % 16 != 0 || (lddo * 2) % 16 != 0) return B200SD_ERR_UNSUPPORTED;
    if (((reinterpret_cast<uintptr_t>(dq) | reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv)) & 15) != 0 ||
        (lddq * 2) % 16 != 0 || (lddk * 2) % 16 != 0 || (lddv * 2) % 16 != 0)
        return B200SD_ERR_UNSUPPORTED;
    BwdTcParams pk, pq;
    memset(&pk, 0, sizeof(pk));
    memset(&pq, 0, sizeof(pq));
    int rc;
    // dK / dV: stationary K, V; streamed Q, dO
    if ((rc = make_map(&pk.tmX1, k, d, heads, (int64_t)batch * Skv, ldk))) return rc;
    if ((rc = make_map(&pk.tmX2, v, d, heads, (int64_t)batch * Skv, ldv))) return rc;
    if ((rc = make_map(&pk.tmY1, q, d, heads, (int64_t)batch * Sq, ldq))) return rc;
    if ((rc = make_map(&pk.tmY2, dout, d, heads, (int64_t)batch * Sq, lddo))) return rc;
    pk.lse = lse; pk.delta = delta; pk.out1 = dv; pk.out2 = dk; pk.Sx = Skv; pk.Sy = Sq; pk.heads = heads; pk.ld1 = lddv; pk.ld2 = lddk;
    pk.scale = scale; pk.scale_log2 = scale * 1.4426950408889634f;
    // dQ: stationary Q, dO; streamed K, V
    if ((rc = make_map(&pq.tmX1, q, d, heads, (int64_t)batch * Sq, ldq))) return rc;
    if ((rc = make_map(&pq.tmX2, dout, d, heads, (int64_t)batch * Sq, lddo))) return rc;
    if ((rc = make_map(&pq.tmY1, k, d, heads, (int64_t)batch * Skv, ldk))) return rc;
    if ((rc = make_map(&pq.tmY2, v, d, heads, (int64_t)batch * Skv, ldv))) return rc;
    pq.lse = lse; pq.delta = delta; pq.out1 = nullptr; pq.out2 = dq; pq.Sx = Sq; pq.Sy = Skv; pq.heads = heads; pq.ld1 = 0; pq.ld2 = lddq;
    pq.scale = scale; pq.scale_log2 = scale * 1.4426950408889634f;
    if (d == 40) {
        if ((rc = launch_one<40, 1, 2, false, true>(pq, batch, s))) return rc;
        return launch_one<40, 1, 2, true, true>(pk, batch, s);
    }
    // d = 80: 2 x 80 accumulator columns leave no room for the TMEM-resident A operands
    if ((rc = launch_one<80, 2, 1, false, false>(pq, batch, s))) return rc;
    return launch_one<80, 2, 1, true, false>(pk, batch, s);
}
