// b200sd -- flash attention on the sm_100a tensor cores (tcgen05 + TMEM): every attention of the SD v1.x UNet -- head dim
// 40 / 80 / 160, self-attention (S_kv = 4096 ... 64) and cross-attention against the 77-token text context (S_kv = 77: the
// second 64-key tile is masked past key 12 before the softmax).  Other head dims keep the register-resident kernel in
// attention.cu.
//
// One CTA = 128 query rows of one (batch, head); it streams 64-key tiles and its softmax warps never wait for the
// tensor core:
//   warp 0    : TMA producer   Q once; K_j, V_j through a 4-stage smem ring (128B-swizzled boxes).  The q/k/v
//               buffers are addressed as 3-D tensors (d, head, row), so a 64-wide box over a 40-wide head is
//               zero-filled past the head by TMA -- no padding kernels, no masking.
//   warp 1    : TMEM allocator + single-thread MMA issuer:
//                   S_j   = Q K_j^T     (M128 x N64, K = d)  -> TMEM, double-buffered: QK^T of tile j+1 is issued before
//                                                              the softmax of tile j has finished
//                   O    += P_j V_j     (M128 x N = d, K = 64), P_j read from TMEM (A operand), O resident in TMEM
//   warps 2-5 : softmax, one thread per query row (its TMEM lane): tcgen05.ld S_j, exp2 in fp32 against a LAGGING
//               reference max (single pass; the tile max is collected on the side), P_j written back to TMEM as bf16
//               (tcgen05.st) -- no shared-memory P tile, no proxy fence.  Only when a row
//               outgrows the reference by 2^kLazyThr is the tile redone (scores are still in registers) and the O
//               rows rescaled in TMEM.  The softmax is MUFU-bound (16 ex2/clk/SM); every 4th score pair is
//               exponentiated on the FMA pipe instead (Cody-Waite + cubic).
// V is consumed in place: its [64 keys x 64 d] TMA boxes are the MN-major B operand of P V (no transpose kernel, no scratch).
// TMEM columns: S0 [0,64)  S1 [64,128)  O [128,128+DN)  P0 P1 [.., +64) (bf16 pairs); two CTAs share an SM at d=40.
// Measured (B200, d=40, S=4096): batch 2 145 -> 117 us, batch 8 480 -> 372 us against the first version (128-key
// tiles, S single-buffered, P through shared memory, O folded in registers every tile, two-pass softmax).
#include <atomic>
#include <cstring>
#include <mutex>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;

namespace {

constexpr int kQ = 128;     // query rows per CTA
constexpr int kBlk = kQ * 128;  // bytes of one [128 rows x 64 bf16] swizzled block

struct AttnParams {
    CUtensorMap tmQ, tmK, tmV;
    bf16* out;
    float* lse;   // optional [batch][heads][Sq]: log2-domain log-sum-exp of the scaled scores (for the backward)
    int Sq, Skv, heads, ldo;
    float scale_log2;
};

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(ptx::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(ptx::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// Blackwell packed fp32x2 math and 3-input max: the softmax warps are instruction-issue bound, these halve the
// non-MUFU instructions per score element (FFMA2 / FADD2 / FMNMX3 in SASS)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
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

// log2 units a row may outgrow the lagging reference max before its tile is redone (P <= 2^6 is harmless in bf16/fp32)
constexpr float kLazyThr = 6.0f;
constexpr int kKV = 64;
constexpr int kThreads = 64 + 4 * 32;   // producer warp, MMA warp, 4 softmax warps
constexpr int kPoly = 4;                // every kPoly-th score pair is exponentiated by poly_exp2x2 instead of MUFU.EX2
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

// 2^t for a pair of scores on the FMA pipe (Cody-Waite split + degree-3 minimax polynomial, 7.5e-5 max relative error --
// P is rounded to bf16, 3.9e-3, right after): the softmax is bound by the 16/clk/SM MUFU unit, so a fraction of the
// exponentials is moved to the idle FMA lanes.  t is clamped to >= -125 so the exponent arithmetic cannot wrap.
__device__ __forceinline__ float2 poly_exp2x2(float2 t) {
    t.x = fmaxf(t.x, -125.f);
    t.y = fmaxf(t.y, -125.f);
    const float2 magic = make_float2(12582912.f, 12582912.f), nmagic = make_float2(-12582912.f, -12582912.f);
    const float2 y = fadd2(t, magic);                      // round-to-nearest integer of t sits in the low mantissa bits
    const float2 ti = fadd2(y, nmagic);
    const float2 f = ffma2(ti, make_float2(-1.f, -1.f), t);   // f = t - round(t) in [-0.5, 0.5]
    float2 q = ffma2(f, make_float2(0.0551716685295105f, 0.0551716685295105f), make_float2(0.2426111251115799f, 0.2426111251115799f));
    q = ffma2(q, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
    q = ffma2(q, f, make_float2(0.9999280571937561f, 0.9999280571937561f));
    float2 e;   // add round(t) to the exponent field: bits(q) + (bits(y) << 23)
    e.x = __uint_as_float((__float_as_uint(y.x) << 23) + __float_as_uint(q.x));   // unsigned: wrap-around is intended
    e.y = __uint_as_float((__float_as_uint(y.y) << 23) + __float_as_uint(q.y));
    return e;
}

// kStages: depth of the K / V smem ring (4; 2 at d = 160, whose three 64-wide d blocks per tile would not fit otherwise)
// Two softmax warps per TMEM lane quadrant (B2 S4096 d40: 129.0 vs 120.9 us) and every exponential on MUFU.EX2 (123.5 vs
// 121.4 us) were measured on B200 and were not faster (DESIGN.md section 5).
template <int D, int DKB, int kStages>
__global__ void __launch_bounds__(kThreads, (D <= 40) ? 2 : 1) attention_tc_kernel(const __grid_constant__ AttnParams p) {
    constexpr int DN = (D + 15) / 16 * 16;    // MMA N of the PV product (48 / 80)
    constexpr int KSTEPS = (D + 15) / 16;     // UMMA K steps of the QK^T product
    constexpr int KBLK = kKV * 128;          // bytes of one K block [64 keys x 64 d]
    constexpr uint32_t kTmemCols = (128 + DN + 64 <= 256) ? 256 : 512;   // S0 S1 | O | P0 P1
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sQ = smem;                               // DKB blocks of [128 q x 64 d]
    uint8_t* sK = sQ + DKB * kBlk;                    // kStages x DKB blocks
    uint8_t* sV = sK + kStages * DKB * KBLK;         // kStages x DKB blocks [64 keys x 64 d]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kStages * DKB * KBLK);
    uint64_t* q_full = bars;
    uint64_t* k_full = bars + 1;                  // [kStages]
    uint64_t* k_empty = k_full + kStages;
    uint64_t* v_full = k_empty + kStages;
    uint64_t* v_empty = v_full + kStages;
    uint64_t* s_full = v_empty + kStages;        // [2]
    uint64_t* p_full = s_full + 2;                // [2]
    uint64_t* o_full = p_full + 2;                // [2]: PV_j commits o_full[j & 1].  Two barriers, because a softmax warp may
                                                  // run one tile ahead of the slowest one: on a single barrier it could find the
                                                  // phase BEFORE the one it waits for still open, which a parity wait cannot tell
                                                  // from "already complete"
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q0 = blockIdx.x * kQ, h = blockIdx.y, b = blockIdx.z;
    const int num_tiles = (p.Skv + kKV - 1) / kKV;   // the last tile may be partial (cross-attention: 77 = 64 + 13 keys)

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&p.tmQ);
        ptx::prefetch_tmap(&p.tmK);
        ptx::prefetch_tmap(&p.tmV);
        ptx::mbar_init(q_full, 1);
        for (int i = 0; i < kStages; ++i) {
            ptx::mbar_init(&k_full[i], 1);
            ptx::mbar_init(&k_empty[i], 1);
            ptx::mbar_init(&v_full[i], 1);
            ptx::mbar_init(&v_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&s_full[i], 1);
            ptx::mbar_init(&p_full[i], 4);    // one (warp-aggregated) arrival per softmax warp
            ptx::mbar_init(&o_full[i], 1);
        }
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
    // P has its own columns: were it written over S (as a first version did), the QK^T of tile j+2 would overwrite columns the
    // PV product of tile j is still reading, ordered by nothing but the tensor pipe's issue order
    const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + 128, tmem_P = tmem_base + 128 + DN;

    if (warp == 0) {
        // ================= TMA producer =================
        if (ptx::elect_one()) {
            ptx::mbar_expect_tx(q_full, DKB * kBlk);
            for (int kb = 0; kb < DKB; ++kb) tma_load_3d(sQ + kb * kBlk, &p.tmQ, q_full, kb * 64, h, b * p.Sq + q0);
            for (int j = 0; j < num_tiles; ++j) {
                const int st = j % kStages;
                const uint32_t ph = (j / kStages) & 1;
                ptx::mbar_wait(&k_empty[st], ph ^ 1);
                ptx::mbar_expect_tx(&k_full[st], DKB * KBLK);
                for (int kb = 0; kb < DKB; ++kb)
                    tma_load_3d(sK + (st * DKB + kb) * KBLK, &p.tmK, &k_full[st], kb * 64, h, b * p.Skv + j * kKV);
                ptx::mbar_wait(&v_empty[st], ph ^ 1);
                ptx::mbar_expect_tx(&v_full[st], DKB * KBLK);
                for (int kb = 0; kb < DKB; ++kb)
                    tma_load_3d(sV + (st * DKB + kb) * KBLK, &p.tmV, &v_full[st], kb * 64, h, b * p.Skv + j * kKV);
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (ptx::elect_one()) {
            const uint32_t idesc_s = ptx::umma_idesc_bf16(128, kKV);
            const uint32_t idesc_o = ptx::umma_idesc_bf16(128, DN) | (1u << 16);   // B (= V, d contiguous) is MN-major
            auto issue_qk = [&](int j) {    // S_j = Q K_j^T into S buffer j & 1
                const int st = j % kStages;
                ptx::mbar_wait(&k_full[st], (j / kStages) & 1);
                ptx::tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < KSTEPS; ++ks) {
                    const int kb = ks / 4, kin = ks % 4;
                    const uint64_t da = ptx::umma_desc_k_sw128(ptx::smem_u32(sQ + kb * kBlk)) + 2 * kin;
                    const uint64_t db = ptx::umma_desc_k_sw128(ptx::smem_u32(sK + (st * DKB + kb) * KBLK)) + 2 * kin;
                    ptx::umma_bf16_ss(tmem_S + (j & 1) * kKV, da, db, idesc_s, ks > 0 ? 1u : 0u);
                }
                ptx::umma_commit(&k_empty[st]);
                ptx::umma_commit(&s_full[j & 1]);
            };
            ptx::mbar_wait(q_full, 0);
            issue_qk(0);
            for (int j = 0; j < num_tiles; ++j) {
                // S buffer (j+1)&1 is free: its last readers were the softmax of tile j-1 (p_full waited below, one
                // iteration ago) and the PV product of tile j-1 (issued earlier on this in-order pipe)
                if (j + 1 < num_tiles) issue_qk(j + 1);
                const int st = j % kStages;
                ptx::mbar_wait(&p_full[j & 1], (j >> 1) & 1);
                ptx::mbar_wait(&v_full[st], (j / kStages) & 1);
                ptx::tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < kKV / 16; ++ks) {   // O += P_j V_j, P read from TMEM (8 columns = 16 keys per step)
                    // 16 keys = two 1024-byte swizzle atoms per k-step; the second 64-wide d block is KBLK further
                    const uint64_t db = ptx::umma_desc_mn_sw128(ptx::smem_u32(sV + st * DKB * KBLK) + ks * 2048, KBLK);
                    ptx::umma_bf16_ts(tmem_O, tmem_P + (j & 1) * 32 + ks * 8, db, idesc_o, (j > 0 || ks > 0) ? 1u : 0u);
                }
                ptx::umma_commit(&v_empty[st]);
                ptx::umma_commit(&o_full[j & 1]);
            }
        }
    } else {
        // ================= softmax warps: one thread per query row =================
        const int qd = warp & 3;                              // TMEM lane quadrant this warp may address
        const int row = qd * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(qd * 32) << 16;
        const uint32_t tO = tmem_O + lane_addr;
        const float2 sc2 = make_float2(p.scale_log2, p.scale_log2);
        float m = -INFINITY, l = 0.f;
        for (int j = 0; j < num_tiles; ++j) {
            const uint32_t tS = tmem_S + lane_addr + (j & 1) * kKV;
            ptx::mbar_wait(&s_full[j & 1], (j >> 1) & 1);
            ptx::tc_fence_after();
            uint32_t r[64], pk[32];
            tmem_ld_32x32b_x32(tS, *reinterpret_cast<uint32_t(*)[32]>(&r[0]));
            tmem_ld_32x32b_x32(tS + 32, *reinterpret_cast<uint32_t(*)[32]>(&r[32]));
            ptx::tmem_ld_wait();
            if ((j + 1) * kKV > p.Skv) {
                // partial last tile: the key rows past S_kv are the next image's keys (or TMA zero fill) -- their scores are
                // set to -inf before the max and the exponentials, so P is exactly 0 there (warp-uniform branch)
                const int valid = p.Skv - j * kKV;
#pragma unroll
                for (int i = 0; i < kKV; ++i)
                    if (i >= valid) r[i] = 0xff800000u;
            }
            // P = exp2(S * scale - off) as packed bf16 pairs; returns the fp32 row sum
            auto exps = [&](float off, bool track, float& mx) -> float {
                const float2 noff2 = make_float2(-off, -off);
                float2 rs2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float2 t = ffma2(make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1])), sc2, noff2);
                    const float2 e = (i % kPoly == kPoly - 1) ? poly_exp2x2(t) : make_float2(fast_exp2(t.x), fast_exp2(t.y));
                    rs2 = fadd2(rs2, e);
                    pk[i] = pack_bf16x2(e.x, e.y);
                    if (track) mx = fmax3(mx, __uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
                }
                return rs2.x + rs2.y;
            };
            float mx = -INFINITY, rs = 0.f;
            bool redo = true;
            if (j > 0) {
                rs = exps(m * p.scale_log2, true, mx);
                redo = __any_sync(0xffffffffu, (mx - m) * p.scale_log2 > kLazyThr);
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) mx = fmax3(mx, __uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
            }
            if (redo) {   // warp-uniform: move every row of the warp to its true running max
                const float mn = fmaxf(m, mx);
                const float corr = fast_exp2((m - mn) * p.scale_log2);
                m = mn;
                float unused = 0.f;
                rs = exps(mn * p.scale_log2, false, unused);
                l *= corr;
                if (j > 0) {   // rescale the O rows accumulated so far (PV_{j-1} must have landed; PV_j waits for p_full)
                    ptx::mbar_wait(&o_full[(j - 1) & 1], ((j - 1) >> 1) & 1);
                    ptx::tc_fence_after();
                    // 48 columns at a time: the scores of this tile stay live in registers (r[64]) across the rescale
#pragma unroll
                    for (int c0 = 0; c0 < DN; c0 += 48) {
                        constexpr int kPiece = 48;
                        uint32_t ob[kPiece];
#pragma unroll
                        for (int c = 0; c < kPiece; c += 16)
                            if (c0 + c < DN) ptx::tmem_ld_32x32b_x16(tO + c0 + c, *reinterpret_cast<uint32_t(*)[16]>(&ob[c]));
                        ptx::tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < kPiece; ++i) ob[i] = __float_as_uint(__uint_as_float(ob[i]) * corr);
#pragma unroll
                        for (int c = 0; c < kPiece; c += 16)
                            if (c0 + c < DN) tmem_st_32x32b_x16(tO + c0 + c, &ob[c]);
                    }
                }
            }
            l += rs;
            // P_j as bf16 pairs into P buffer j & 1: its previous reader, PV_{j-2}, completed before QK_j did (s_full above)
            const uint32_t tP = tmem_P + lane_addr + (j & 1) * 32;
            tmem_st_32x32b_x16(tP, &pk[0]);
            tmem_st_32x32b_x16(tP + 16, &pk[16]);
            ptx::tmem_st_wait();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&p_full[j & 1]);
        }
        // ---- normalise and store ----
        ptx::mbar_wait(&o_full[(num_tiles - 1) & 1], ((num_tiles - 1) >> 1) & 1);
        ptx::tc_fence_after();
        const float inv = 1.0f / l;
        const bool live = q0 + row < p.Sq;   // S_q tail: rows past the image's last query were computed on foreign rows -- not stored
        if (p.lse != nullptr && live) p.lse[((size_t)b * p.heads + h) * p.Sq + q0 + row] = m * p.scale_log2 + log2f(l);
        bf16* dst = p.out + ((size_t)b * p.Sq + q0 + row) * p.ldo + h * D;
#pragma unroll
        for (int c0 = 0; c0 < DN; c0 += 16) {
            uint32_t ob[16];
            ptx::tmem_ld_32x32b_x16(tO + c0, ob);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 16; c += 8) {
                if (c0 + c < D && live) {
                    uint4 u;
                    u.x = pack_bf16x2(__uint_as_float(ob[c]) * inv, __uint_as_float(ob[c + 1]) * inv);
                    u.y = pack_bf16x2(__uint_as_float(ob[c + 2]) * inv, __uint_as_float(ob[c + 3]) * inv);
                    u.z = pack_bf16x2(__uint_as_float(ob[c + 4]) * inv, __uint_as_float(ob[c + 5]) * inv);
                    u.w = pack_bf16x2(__uint_as_float(ob[c + 6]) * inv, __uint_as_float(ob[c + 7]) * inv);
                    *reinterpret_cast<uint4*>(dst + c0 + c) = u;
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

template <int D, int DKB, int kStages>
int launch_tc(const bf16* q, const bf16* k, const bf16* v, bf16* out, float* lse, int batch, int heads, int Sq, int Skv, int ldq,
               int ldk, int ldv, int ldo, float scale, cudaStream_t s) {
    AttnParams p;
    memset(&p, 0, sizeof(p));
    {
        const uint64_t dims[3] = {(uint64_t)D, (uint64_t)heads, (uint64_t)batch * Sq};
        const uint64_t str[3] = {0, (uint64_t)D * 2, (uint64_t)ldq * 2};
        const uint32_t box[3] = {64, 1, 128};
        int rc = b200sd_make_tmap(&p.tmQ, q, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }
    {
        const uint64_t dims[3] = {(uint64_t)D, (uint64_t)heads, (uint64_t)batch * Skv};
        const uint64_t str[3] = {0, (uint64_t)D * 2, (uint64_t)ldk * 2};
        const uint32_t box[3] = {64, 1, (uint32_t)kKV};
        int rc = b200sd_make_tmap(&p.tmK, k, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }
    {
        const uint64_t dims[3] = {(uint64_t)D, (uint64_t)heads, (uint64_t)batch * Skv};
        const uint64_t str[3] = {0, (uint64_t)D * 2, (uint64_t)ldv * 2};
        const uint32_t box[3] = {64, 1, (uint32_t)kKV};
        int rc = b200sd_make_tmap(&p.tmV, v, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }
    p.out = out;
    p.lse = lse;
    p.Sq = Sq;
    p.Skv = Skv;
    p.heads = heads;
    p.ldo = ldo;
    p.scale_log2 = scale * 1.4426950408889634f;
    const size_t smem = (size_t)DKB * kBlk + (size_t)2 * kStages * DKB * kKV * 128 + 256 + 1024;
    B200SD_CUDA(b200sd_opt_in_smem(attention_tc_kernel<D, DKB, kStages>, (int)smem, /*max_carveout=*/true));
    attention_tc_kernel<D, DKB, kStages><<<dim3((Sq + kQ - 1) / kQ, heads, batch), dim3(kThreads), smem, s>>>(p);
    g_b200sd_launches.fetch_add(1, std::memory_order_relaxed);
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

}  // namespace

// Returns B200SD_ERR_UNSUPPORTED when the shape is not covered (the caller falls back to attention.cu's kernel).
int b200sd_attention_tc(const void* q, const void* k, const void* v, void* out, float* lse, int batch, int heads, int Sq, int Skv,
                        int d, int ldq, int ldk, int ldv, int ldo, float scale, void* workspace, size_t ws_bytes,
                        cudaStream_t s) {
    if (!(d == 40 || d == 80 || d == 160) || Sq < 1 || Skv < 1) return B200SD_ERR_UNSUPPORTED;
    (void)workspace;   // no scratch any more: V is consumed in place (MN-major B operand), the V^T transpose kernel is gone
    (void)ws_bytes;
    if ((ldq * 2) % 16 != 0 || (ldk * 2) % 16 != 0 || (ldv * 2) % 16 != 0) return B200SD_ERR_UNSUPPORTED;
    const bf16 *qb = static_cast<const bf16*>(q), *kb = static_cast<const bf16*>(k), *vb = static_cast<const bf16*>(v);
    bf16* ob = static_cast<bf16*>(out);
    if (d == 40) return launch_tc<40, 1, 4>(qb, kb, vb, ob, lse, batch, heads, Sq, Skv, ldq, ldk, ldv, ldo, scale, s);
    if (d == 80) return launch_tc<80, 2, 4>(qb, kb, vb, ob, lse, batch, heads, Sq, Skv, ldq, ldk, ldv, ldo, scale, s);
    return launch_tc<160, 3, 2>(qb, kb, vb, ob, lse, batch, heads, Sq, Skv, ldq, ldk, ldv, ldo, scale, s);
}
