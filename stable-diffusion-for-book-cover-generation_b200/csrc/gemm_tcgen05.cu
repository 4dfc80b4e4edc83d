// b200sd -- GEMM / implicit-GEMM 3x3 convolution on the sm_100a tensor cores.
//
//   out[M, N] = A[M, K] * W[N, K]^T (+ bias) (+ rowbias) (+ residual)     bf16 x bf16 -> fp32 -> bf16
//
// Warp-specialised, one 128 x BLOCK_N output tile (x one K split) per CTA:
//   warp 0      : TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier full/empty)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (accumulator in TMEM)
//   warps 2..5  : epilogue (tcgen05.ld TMEM -> registers -> fused bias/temb/residual/GEGLU -> global)
// 3x3 convolution is the same pipeline with the A operand gathered by 4-D TMA boxes over the NHWC
// activation: one (64 ch, W, rows, images) box per (tap, 64-channel block); the +-1 halo of the
// padding comes from TMA out-of-bounds zero fill, so no im2col buffer ever exists.  A second
// activation source (a1) extends the channel axis, which fuses the up-block torch.cat.
// With <= 113 KB of smem and <= 256 TMEM columns per CTA two CTAs share an SM, so one CTA's
// epilogue overlaps the other's main loop.  Small-M / deep-K layers are split along K with a
// the split CTAs of a tile form a thread-block cluster, exchange their fp32 partial tiles through
// distributed shared memory, and each reduces + stores 128/split rows in a fixed order (deterministic).
#include <atomic>
#include <cstring>
#include <mutex>
#include <cstdio>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;

// debug override (tools/cold_probe.py): key 0 = persistent kernel (-1 default, 0 off, 1 on)
static int g_persist = -1;
extern "C" void b200sd_debug_set(int key, int value) { if (key == 0) g_persist = value; }

namespace {

constexpr int BLOCK_M = 128;
constexpr size_t kWsPartialBytes = (size_t)160 * 128 * 256 * sizeof(float);   // split-K partial tiles (<= one per SM), see b200sd_gemm_workspace_bytes
constexpr size_t kWsCounterBytes = 4096;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int kNumThreads = 192;
constexpr int kMaxStages = 8;
constexpr int kABytes = BLOCK_M * BLOCK_K * 2;  // 16 KB (always reserved in full)


struct KParams {
    CUtensorMap tmA0, tmA1, tmB;
    const float* bias;
    const float* rowbias;
    const void* residual;
    void* out;
    int M, N;
    int num_k_blocks;    // total K / 64
    int kb_per_split;
    int split_k;
    int block_n;
    int stages;
    int conv;            // 0 plain, 1 conv3x3
    int cblocks0;        // C0 / 64
    int cblocks;         // (C0 + C1) / 64
    int tile_w, tile_h, tile_n;   // conv box geometry
    int tiles_y;         // H / tile_h (conv, tile_n == 1)
    int tiles_x;         // W / tile_w: 1 unless an image row is wider than one 128-pixel tile (VAE: W = 256 / 512)
    int rows_valid;      // valid rows in a tile (<= 128)
    int a_bytes;         // bytes TMA delivers for A per stage
    int ldc, ldr, ldrb;
    int rows_per_image;
    int epilogue;
    int out_f32;
    int res_f32;
    uint32_t tmem_cols;
    // ---- backward (dgrad / wgrad) operand modes ----
    int a_mn;            // 1: A is MN-major (wgrad: A = dY [rows = K][M channels]), two 64-channel boxes per stage
    int b_mode;          // 0 K-major [N][K]; 1 MN-major weights [K][N] (dgrad; 3-D (ci, tap, co) for conv);
                         // 2 MN-major activations [rows = K][N] (wgrad); 3 same, 3x3-shifted 4-D boxes (conv wgrad)
    int conv_sign;       // +1 forward taps, -1 dgrad (A sampled at p - d(tap))
    int n_valid;         // output columns that exist (tiles may overhang when block_n does not divide N)
    int tiles_per_tap;   // conv wgrad: n-tiles per tap (output column = tap * n_valid + c)
    int atomic_out;      // fp32 red.add into `out` (wgrad: split-K partials and gradient accumulation)
    int pair;            // CTA pair (cta_group::2): two CTAs adjacent in M form one 256 x block_n MMA tile; each loads its own
                         // 128 A rows and HALF of the B tile, so the L2 -> smem traffic per FLOP drops by ~1/3
    int persist;         // host only: this launch goes to gemm_persist_kernel (set by gemm_tiling)
    int psplit;          // host only: ... in its split-K mode with this many K slices per tile (0 = no)
    float* gn_part;      // optional [m_tiles * split_k][2][N]: per-column (sum, sum of squares) of the rows each CTA stores --
                         // the GroupNorm that consumes this output gets its statistics from here instead of re-reading it
};

// cluster helpers (split-K reduction over distributed shared memory)
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ float4 ld_dsmem_v4(uint32_t local_smem_addr, uint32_t cta_rank) {
    uint32_t raddr;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(local_smem_addr), "r"(cta_rank));
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(raddr) : "memory");
    return v;
}

__device__ __forceinline__ void red_add_v4(float* dst, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---- store phase of the epilogue: one thread = one 8-column group, walking down the rows of the staging tile ----
struct EpiCtx {
    uint32_t stage_u32;
    int pitch_f, row_end, R, cb, half, m0, col_out, img0, n0cb;
    const float* s_rb;
    bool multi_img, rb_smem;
};
__device__ __forceinline__ void lds8(uint32_t addr, float (&v)[8]) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(addr + 16));
}
// OUT: 0 bf16, 1 fp32, 2 fp32 red.add;  RES: 0 none, 1 bf16, 2 fp32;  SPLIT: sum the cluster's partial tiles over DSMEM
// STATS: also accumulate this thread's per-column sum / sum of squares of the values it stores (cs / cq)
template <int OUT, int RES, bool SPLIT, bool GEGLU, bool STATS = false>
__device__ __forceinline__ void epilogue_rows(const KParams& p, const EpiCtx& e, int row0, const float (&b)[8], const float (&bg)[8],
                                              float* cs = nullptr, float* cq = nullptr) {
    constexpr int U = 4;
    for (int row = row0; row < e.row_end; row += e.R * U) {
        float v[U][8], r[U][8];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int rl = min(row + u * e.R, e.row_end - 1);   // clamped: loads of a masked-off row stay in bounds
            const uint32_t addr = e.stage_u32 + (uint32_t)(rl * e.pitch_f + e.cb) * 4u;
            if constexpr (SPLIT) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[u][i] = 0.f;
                for (int sp = 0; sp < p.split_k; ++sp) {
                    const float4 a0 = ld_dsmem_v4(addr, sp), a1 = ld_dsmem_v4(addr + 16, sp);
                    v[u][0] += a0.x; v[u][1] += a0.y; v[u][2] += a0.z; v[u][3] += a0.w;
                    v[u][4] += a1.x; v[u][5] += a1.y; v[u][6] += a1.z; v[u][7] += a1.w;
                }
            } else {
                lds8(addr, v[u]);
            }
            if constexpr (GEGLU) lds8(addr + (uint32_t)e.half * 4u, r[u]);
            else if constexpr (RES == 2) ld8<B200SD_F32>(p.residual, (size_t)(e.m0 + rl) * p.ldr + e.col_out, r[u]);
            else if constexpr (RES == 1) ld8<B200SD_BF16>(p.residual, (size_t)(e.m0 + rl) * p.ldr + e.col_out, r[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int rl = row + u * e.R;
            if (rl >= e.row_end) break;
            const int grow = e.m0 + rl;
            float o[8];
            if constexpr (GEGLU) {
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = (v[u][i] + b[i]) * gelu_erf_f(r[u][i] + bg[i]);
                st8<B200SD_BF16>(p.out, (size_t)grow * p.ldc + e.col_out, o);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = v[u][i] + b[i];
                if constexpr (RES != 0) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) o[i] += r[u][i];
                }
                if (e.multi_img) {   // tile spans several images (8x8 / 4x4 levels): per-row time-embedding bias
                    const int img = grow / p.rows_per_image;
                    if (e.rb_smem) {
                        const float* rb = e.s_rb + (img == e.img0 ? 0 : 256) + e.cb;
#pragma unroll
                        for (int i = 0; i < 8; ++i) o[i] += rb[i];
                    } else {
                        float t[8];
                        ld8<B200SD_F32>(p.rowbias, (size_t)img * p.ldrb + e.n0cb, t);
#pragma unroll
                        for (int i = 0; i < 8; ++i) o[i] += t[i];
                    }
                }
                if constexpr (STATS) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) { cs[i] += o[i]; cq[i] = fmaf(o[i], o[i], cq[i]); }
                }
                if constexpr (OUT == 2) {
                    float* dst = static_cast<float*>(p.out) + (size_t)grow * p.ldc + e.col_out;
                    red_add_v4(dst, o[0], o[1], o[2], o[3]);
                    red_add_v4(dst + 4, o[4], o[5], o[6], o[7]);
                } else if constexpr (OUT == 1) st8<B200SD_F32>(p.out, (size_t)grow * p.ldc + e.col_out, o);
                else st8<B200SD_BF16>(p.out, (size_t)grow * p.ldc + e.col_out, o);
            }
        }
    }
}

// PAIR is a compile-time switch: a kernel that contains cta_group::2 instructions can only be launched as CTA pairs
// OP selects the operand modes at compile time (0 forward: both K-major; 1 dgrad: B = weights MN-major; 2 / 3 wgrad
// plain / conv3x3: A and B MN-major), so the forward instantiation carries none of the backward's branches.
template <bool PAIR, int OP>
__global__ void __launch_bounds__(kNumThreads, 1) gemm_tcgen05_kernel(const __grid_constant__ KParams p) {
    constexpr bool a_mn = OP >= 2;
    constexpr int b_mode = OP;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment for the 128B swizzle atoms
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr bool pair = PAIR;
    const uint32_t crank = pair ? cluster_ctarank() : 0;          // pair = cluster (2,1,1): rank 0 is the MMA leader
    const int b_bytes = (p.block_n * BLOCK_K * 2) >> (pair ? 1 : 0);   // B bytes held by THIS CTA per stage
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + (size_t)p.stages * kABytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)p.stages * b_bytes);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kMaxStages;
    uint64_t* tmem_full_bar = bars + 2 * kMaxStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x;
    const int n_tile = blockIdx.y;
    const int split = blockIdx.z;
    const int kb_begin = split * p.kb_per_split;
    const int kb_end = min(kb_begin + p.kb_per_split, p.num_k_blocks);
    // conv wgrad: the N axis is (tap, input channel); a tile never straddles taps
    const int w_tap = b_mode == 3 ? n_tile / p.tiles_per_tap : 0;
    const int n0 = (b_mode == 3 ? n_tile - w_tap * p.tiles_per_tap : n_tile) * p.block_n;   // column within the (per-tap) N axis
    const int col_base = w_tap * p.n_valid + n0;                                             // output column of tile column 0
    const int col_valid = min(p.block_n, p.n_valid - n0);
    const int m0 = m_tile * p.rows_valid;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&p.tmA0);
        ptx::prefetch_tmap(&p.tmB);
        if (p.cblocks0 != p.cblocks) ptx::prefetch_tmap(&p.tmA1);
        for (int s = 0; s < p.stages; ++s) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        ptx::mbar_init(tmem_full_bar, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        if constexpr (pair) { ptx::tmem_alloc_cg2(tmem_slot, p.tmem_cols); ptx::tmem_relinquish_cg2(); }
        else { ptx::tmem_alloc(tmem_slot, p.tmem_cols); ptx::tmem_relinquish(); }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (pair) cluster_sync_all();   // the peer's barriers must be initialised before anything is signalled on them
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // epilogue-side shared state (also visible to part 2 after the role dispatch)
    const int epi_tid = threadIdx.x - 64;  // 0..127 for the epilogue warps
    const int pitch_f = p.block_n + 4;     // +16 B: conflict-free 16-byte row-strided stores
    float* stage = reinterpret_cast<float*>(smem);
    float* s_bias = reinterpret_cast<float*>(bars + 32);   // [256]
    float* s_rb = s_bias + 256;                            // [2][256] row-bias of the (at most two) images of this tile
    int img0 = 0, img1 = 0;
    bool rb_smem = false;
    if (p.rowbias && m0 < p.M) {
        img0 = m0 / p.rows_per_image;
        img1 = (min(m0 + p.rows_valid, p.M) - 1) / p.rows_per_image;
        rb_smem = (img1 - img0) <= 1;
    }

    if (warp == 0) {
        // ================= TMA producer =================
        if (ptx::elect_one()) {
            int stage = 0;
            uint32_t phase = 0;
            int img = 0, y0 = 0, x0 = 0;
            if (p.conv) {
                if (p.tile_n > 1) { img = m_tile * p.tile_n; y0 = 0; }
                else {
                    int mt = m_tile;
                    if (p.tiles_x > 1) { x0 = (mt % p.tiles_x) * p.tile_w; mt /= p.tiles_x; }
                    img = mt / p.tiles_y; y0 = (mt % p.tiles_y) * p.tile_h;
                }
            }
            // pair mode: this CTA loads its own A rows and half of the B tile; completion is signalled on the leader's barrier
            // MN-major B: only the 64-column boxes that hold existing columns are loaded (the last N tile of a layer may be
            // narrower than block_n: N = 320 runs as 192 + 128); a pair splits the full tile evenly and keeps it whole
            const int nbox_live = (b_mode != 0 && !pair) ? (col_valid + 63) >> 6 : (p.block_n >> 6);
            const int nboxb = nbox_live >> (pair ? 1 : 0);   // 64-column boxes of an MN-major B tile held by this CTA
            const int nb0 = n0 + (pair ? (int)crank * (p.block_n >> 1) : 0);
            const uint32_t stage_tx = (b_mode != 0 && !pair) ? (uint32_t)(p.a_bytes + nbox_live * 8192)
                                                             : ((uint32_t)(p.a_bytes + b_bytes) << (pair ? 1 : 0));
            for (int kb = kb_begin; kb < kb_end; ++kb) {
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                if (!pair || crank == 0) ptx::mbar_expect_tx(&full_bar[stage], stage_tx);
                uint8_t* dst_a = smem_a + (size_t)stage * kABytes;
                uint8_t* dst_b = smem_b + (size_t)stage * b_bytes;
                uint64_t* fb = &full_bar[stage];
                const uint32_t fbc = pair ? ptx::mapa_u32(ptx::smem_u32(fb), 0) : 0;
#define LD2(dst, tm, c0, c1) do { if constexpr (pair) ptx::tma_load_2d_cg2(dst, tm, fbc, c0, c1); else ptx::tma_load_2d(dst, tm, fb, c0, c1); } while (0)
#define LD3(dst, tm, c0, c1, c2) do { if constexpr (pair) ptx::tma_load_3d_cg2(dst, tm, fbc, c0, c1, c2); else ptx::tma_load_3d(dst, tm, fb, c0, c1, c2); } while (0)
#define LD4(dst, tm, c0, c1, c2, c3) do { if constexpr (pair) ptx::tma_load_4d_cg2(dst, tm, fbc, c0, c1, c2, c3); else ptx::tma_load_4d(dst, tm, fb, c0, c1, c2, c3); } while (0)
                // ---- A ----
                if (a_mn) {
                    LD2(dst_a, &p.tmA0, m0, kb * BLOCK_K);
                    LD2(dst_a + kABytes / 2, &p.tmA0, m0 + 64, kb * BLOCK_K);
                } else if (!p.conv) {
                    if (kb < p.cblocks0) LD2(dst_a, &p.tmA0, kb * BLOCK_K, m0);
                    else LD2(dst_a, &p.tmA1, (kb - p.cblocks0) * BLOCK_K, m0);
                } else {
                    const int tap = kb / p.cblocks;
                    const int cb = kb - tap * p.cblocks;
                    const int dy = (tap / 3 - 1) * p.conv_sign, dx = (tap % 3 - 1) * p.conv_sign;
                    if (cb < p.cblocks0) LD4(dst_a, &p.tmA0, cb * BLOCK_K, x0 + dx, y0 + dy, img);
                    else LD4(dst_a, &p.tmA1, (cb - p.cblocks0) * BLOCK_K, x0 + dx, y0 + dy, img);
                }
                // ---- B ----
                if (b_mode == 0) {
                    LD2(dst_b, &p.tmB, kb * BLOCK_K, nb0);
                } else if (b_mode == 1) {
                    if (!p.conv) {
                        for (int j = 0; j < nboxb; ++j) LD2(dst_b + j * 8192, &p.tmB, nb0 + j * 64, kb * BLOCK_K);
                    } else {
                        const int tap = kb / p.cblocks;
                        const int cb = kb - tap * p.cblocks;
                        for (int j = 0; j < nboxb; ++j) LD3(dst_b + j * 8192, &p.tmB, nb0 + j * 64, tap, cb * BLOCK_K);
                    }
                } else if (b_mode == 2) {
                    for (int j = 0; j < nboxb; ++j) LD2(dst_b + j * 8192, &p.tmB, nb0 + j * 64, kb * BLOCK_K);
                } else {
                    // conv wgrad: k-block kb = 64 pixels = box (64 ch, W, tile_h, tile_n) shifted by the tap
                    int bimg, by0;
                    if (p.tile_n > 1) { bimg = kb * p.tile_n; by0 = 0; }
                    else { bimg = kb / p.tiles_y; by0 = (kb - bimg * p.tiles_y) * p.tile_h; }
                    const int dy = w_tap / 3 - 1, dx = w_tap % 3 - 1;
                    for (int j = 0; j < nboxb; ++j) LD4(dst_b + j * 8192, &p.tmB, nb0 + j * 64, dx, by0 + dy, bimg);
                }
#undef LD2
#undef LD3
#undef LD4
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (one elected thread) =================
        if ((!pair || crank == 0) && ptx::elect_one()) {
            const uint32_t b_mn = b_mode != 0;
            const uint32_t mma_n = (b_mode != 0 && !pair) ? (uint32_t)(((col_valid + 63) >> 6) << 6) : (uint32_t)p.block_n;   // live boxes only
            const uint32_t idesc = ptx::umma_idesc_bf16(pair ? 2 * BLOCK_M : BLOCK_M, mma_n) | ((uint32_t)a_mn << 15) | (b_mn << 16);
            // K-major: +32 B per UMMA_K inside the swizzle atom; MN-major: 16 k-rows = two 1024-byte atoms further
            const uint32_t a_step = a_mn ? (2048 >> 4) : 2, b_step = b_mn ? (2048 >> 4) : 2;
            int stage = 0;
            uint32_t phase = 0;
            for (int kb = kb_begin; kb < kb_end; ++kb) {
                ptx::mbar_wait(&full_bar[stage], phase);
                ptx::tc_fence_after();
                const uint32_t sa = ptx::smem_u32(smem_a + (size_t)stage * kABytes), sb = ptx::smem_u32(smem_b + (size_t)stage * b_bytes);
                const uint64_t da = a_mn ? ptx::umma_desc_mn_sw128(sa, 8192) : ptx::umma_desc_k_sw128(sa);
                const uint64_t db = b_mn ? ptx::umma_desc_mn_sw128(sb, 8192) : ptx::umma_desc_k_sw128(sb);
#pragma unroll
                for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                    const uint32_t accum = (kb > kb_begin || k > 0) ? 1u : 0u;
                    if constexpr (pair) ptx::umma_bf16_ss_cg2(tmem_base, da + a_step * k, db + b_step * k, idesc, accum);
                    else ptx::umma_bf16_ss(tmem_base, da + a_step * k, db + b_step * k, idesc, accum);
                }
                // frees the smem slot (of both CTAs in pair mode) when these MMAs retire
                if constexpr (pair) ptx::umma_commit_cg2(&empty_bar[stage], 3); else ptx::umma_commit(&empty_bar[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            if constexpr (pair) ptx::umma_commit_cg2(tmem_full_bar, 3); else ptx::umma_commit(tmem_full_bar);
        }
    } else {
        // ================= epilogue warps, part 1 =================
        // While the main loop runs: park this tile's bias (and time-embedding row bias) in smem.
        // Then TMEM -> registers -> fp32 staging tile in the (by then idle) smem ring, one row per thread.
        const int q = warp & 3;              // TMEM lane quarter this warp may access
        const int r_in_tile = q * 32 + lane;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        for (int c = epi_tid; c < p.block_n; c += 128) {
            s_bias[c] = (p.bias && c < col_valid) ? __ldg(p.bias + n0 + c) : 0.f;
            if (rb_smem) {
                s_rb[c] = __ldg(p.rowbias + (size_t)img0 * p.ldrb + n0 + c);
                s_rb[256 + c] = __ldg(p.rowbias + (size_t)img1 * p.ldrb + n0 + c);
            }
        }
        ptx::mbar_wait(tmem_full_bar, 0);
        ptx::tc_fence_after();
        {
            float4* my_row = reinterpret_cast<float4*>(stage + (size_t)r_in_tile * pitch_f);
            for (int c = 0; c < p.block_n; c += 32) {
                uint32_t r0[16], r1[16];
                const bool two = (c + 16 < p.block_n);
                ptx::tmem_ld_32x32b_x16(taddr + c, r0);
                if (two) ptx::tmem_ld_32x32b_x16(taddr + c + 16, r1);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    my_row[c / 4 + i] = make_float4(__uint_as_float(r0[4 * i]), __uint_as_float(r0[4 * i + 1]),
                                                    __uint_as_float(r0[4 * i + 2]), __uint_as_float(r0[4 * i + 3]));
                if (two) {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        my_row[c / 4 + 4 + i] = make_float4(__uint_as_float(r1[4 * i]), __uint_as_float(r1[4 * i + 1]),
                                                            __uint_as_float(r1[4 * i + 2]), __uint_as_float(r1[4 * i + 3]));
                }
            }
        }
        ptx::tc_fence_before();
        ptx::named_bar_sync(1, 128);  // whole staging tile (and the bias tiles) written
    }

    // Split-K: the `split_k` CTAs of a tile form one thread-block cluster; after this barrier every CTA can
    // read its peers' staging tiles through distributed shared memory.  Otherwise a CTA barrier: ALL warps
    // (the producer and MMA warps are done by now) take part in the store phase.
    if (p.split_k > 1) cluster_sync_all(); else __syncthreads();

    {
        // ================= epilogue, part 2: reduce (split-K) + fused epilogue + coalesced stores =================
        // Every thread owns ONE 8-column group of the tile and walks down the rows (R rows per pass, U passes in
        // flight): no index arithmetic in the loop, bias in registers, consecutive threads on consecutive 16/32-byte
        // vectors of a row.  With split-K each CTA of the cluster owns 128/split_k rows and sums the split partials
        // in a fixed order (deterministic).  Loads of a batch are issued before any store so that (possibly
        // aliasing, in-place) residual reads are not serialised behind the stores.
        const int rank = p.split_k > 1 ? (int)cluster_ctarank() : 0;
        const int rows_per_cta = BLOCK_M / p.split_k;
        const int row_begin = rank * rows_per_cta;
        int valid = min(p.rows_valid, p.M - m0) - row_begin;
        valid = max(0, min(valid, rows_per_cta));
        const bool geglu = p.epilogue == B200SD_EPI_GEGLU;
        const int half = p.block_n / 2;
        const int groups = (geglu ? half : p.block_n) / 8;
        const int R = kNumThreads / groups;           // rows per pass
        const int tid = threadIdx.x;
        float cs[8], cq[8];   // GroupNorm column statistics of the rows this thread stores (p.gn_part)
#pragma unroll
        for (int i = 0; i < 8; ++i) { cs[i] = 0.f; cq[i] = 0.f; }
        if (tid < R * groups && valid > 0) {
            const int c8 = tid % groups, r0 = tid / groups;
            const int cb = c8 * 8;
            if (geglu || cb < col_valid) {
                float b[8], bg[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { b[i] = s_bias[cb + i]; bg[i] = geglu ? s_bias[half + cb + i] : 0.f; }
                const bool multi_img = p.rowbias != nullptr && img1 != img0;
                if (p.rowbias != nullptr && !multi_img) {   // one image per tile (the common case): fold the time embedding into the bias
#pragma unroll
                    for (int i = 0; i < 8; ++i) b[i] += s_rb[cb + i];
                }
                EpiCtx e;
                e.stage_u32 = ptx::smem_u32(stage);
                e.pitch_f = pitch_f; e.row_end = row_begin + valid; e.R = R; e.cb = cb; e.half = half; e.m0 = m0;
                e.col_out = geglu ? n_tile * half + cb : col_base + cb;
                e.s_rb = s_rb; e.img0 = img0; e.multi_img = multi_img; e.rb_smem = rb_smem; e.n0cb = n0 + cb;
                const int row0 = row_begin + r0;
                const int ok = p.atomic_out ? 2 : (p.out_f32 ? 1 : 0);
                const int rk = p.residual ? (p.res_f32 ? 2 : 1) : 0;
                if (geglu) epilogue_rows<0, 0, false, true>(p, e, row0, b, bg);
                else if (p.split_k > 1) {
                    if (ok == 1 && p.gn_part) { if (rk == 2) epilogue_rows<1, 2, true, false, true>(p, e, row0, b, bg, cs, cq); else epilogue_rows<1, 0, true, false, true>(p, e, row0, b, bg, cs, cq); }
                    else if (ok == 1) { if (rk == 2) epilogue_rows<1, 2, true, false>(p, e, row0, b, bg); else if (rk == 1) epilogue_rows<1, 1, true, false>(p, e, row0, b, bg); else epilogue_rows<1, 0, true, false>(p, e, row0, b, bg); }
                    else { if (rk == 2) epilogue_rows<0, 2, true, false>(p, e, row0, b, bg); else if (rk == 1) epilogue_rows<0, 1, true, false>(p, e, row0, b, bg); else epilogue_rows<0, 0, true, false>(p, e, row0, b, bg); }
                } else if (ok == 2) epilogue_rows<2, 0, false, false>(p, e, row0, b, bg);
                else if (ok == 1 && p.gn_part) { if (rk == 2) epilogue_rows<1, 2, false, false, true>(p, e, row0, b, bg, cs, cq); else epilogue_rows<1, 0, false, false, true>(p, e, row0, b, bg, cs, cq); }
                else if (ok == 1) { if (rk == 2) epilogue_rows<1, 2, false, false>(p, e, row0, b, bg); else if (rk == 1) epilogue_rows<1, 1, false, false>(p, e, row0, b, bg); else epilogue_rows<1, 0, false, false>(p, e, row0, b, bg); }
                else { if (rk == 2) epilogue_rows<0, 2, false, false>(p, e, row0, b, bg); else if (rk == 1) epilogue_rows<0, 1, false, false>(p, e, row0, b, bg); else epilogue_rows<0, 0, false, false>(p, e, row0, b, bg); }
            }
        }
        if (p.gn_part != nullptr) {
            // GroupNorm statistics of the rows this CTA stored.  Once nobody reads the staging tile any more (peers included),
            // it becomes the scratch for a fixed-order (deterministic) fold of the R row-walkers of every column group;
            // partial row (m_tile * split_k + rank) = [sum | sum of squares][N].
            if (p.split_k > 1) cluster_sync_all(); else __syncthreads();
            float* s_gn = reinterpret_cast<float*>(stage);
#pragma unroll
            for (int i = 0; i < 8; ++i) { s_gn[tid * 16 + i] = cs[i]; s_gn[tid * 16 + 8 + i] = cq[i]; }
            __syncthreads();
            float* dst = p.gn_part + (size_t)(m_tile * p.split_k + rank) * 2 * p.N;
            for (int idx = tid; idx < groups * 16; idx += kNumThreads) {
                const int c8 = idx >> 4, k = idx & 15, col = c8 * 8 + (k & 7);
                float a = 0.f;
                for (int r = 0; r < R; ++r) a += s_gn[(r * groups + c8) * 16 + k];
                if (col < col_valid) dst[(size_t)(k >> 3) * p.N + n0 + col] = a;
            }
        }
    }
    // peers may still be reading this CTA's staging tile (with gn_part the cluster has already synchronised above)
    if (p.split_k > 1 && p.gn_part == nullptr) cluster_sync_all();

    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (pair) cluster_sync_all();   // the leader's MMAs read the peer's smem / write its TMEM: nobody leaves early
    if (warp == 1) {
        ptx::tc_fence_after();
        if constexpr (pair) ptx::tmem_dealloc_cg2(tmem_base, p.tmem_cols); else ptx::tmem_dealloc(tmem_base, p.tmem_cols);
    }
}

// =================================================================================================================
// Persistent forward kernel: one CTA per SM walks the output tiles of the layer (tile = blockIdx.x + i * gridDim.x).
//   warp 0     : TMA producer -- runs ahead across tile boundaries, the smem ring never drains between tiles
//   warp 1     : TMEM allocator + tcgen05.mma issuer; TWO accumulator stages in TMEM, so the MMAs of tile i+1 are issued
//                while the epilogue warps still drain tile i
//   warps 2..9 : epilogue, TWO warps per 32-lane quarter of the accumulator (a warp may only touch the TMEM lanes of its
//                quarter = 32 output rows); the pair splits the tile's 32-column chunks odd / even.  Per chunk: tcgen05.ld -> registers -> (+bias, +time embedding, +residual | GEGLU) -> swizzled
//                4 KB smem chunk -> TMA store (cp.async.bulk.tensor, bulk groups).  The residual chunk arrives by TMA in
//                the SAME smem chunk, issued `depth - 1` chunks ahead (for a one-tile CTA: during the main loop), so no
//                epilogue thread ever waits on a global load -- the old store phase was bound by exactly that latency
//                (7 of the 10.7 us of an M8192 N320 K320 projection).
// GroupNorm column statistics (gn_part) are summed from the finished fp32 chunk in smem, one partial row per (tile, warp).
// Covers forward GEMM / conv3x3 tiles of 128 rows without split-K and without CTA pairs; everything else stays on
// gemm_tcgen05_kernel above.
// =================================================================================================================
constexpr int kEpiWarps = 8;
constexpr int kPersistThreads = 64 + 32 * kEpiWarps + 32;   // A producer | MMA | 8 epilogue | B producer
constexpr int kMaxDepth = 3;

struct PParams {
    CUtensorMap tmA0, tmA1, tmB, tmOut, tmRes;
    const float* bias;
    const float* rowbias;
    float* gn_part;
    int M, N;
    int num_k_blocks, block_n, stages;
    int conv, cblocks0, cblocks, tile_h, tile_n, tiles_y;
    int tile_w, tiles_x;            // image rows wider than a tile (see KParams::tiles_x)
    int n_tiles, num_tiles;
    int ldrb, rows_per_image;
    int geglu, out_f32, res_kind;   // res_kind: 0 none, 1 bf16, 2 fp32
    int depth;                      // smem chunks per epilogue warp (3 with a residual, 2 without)
    int chunk_bytes;                // 4096: 32 rows x 128 B (an fp32 chunk is involved); 2048: 32 rows x 64 B (bf16 only)
    uint32_t tmem_cols, acc_stride;
    uint32_t off_b, off_epi, off_bias, off_stat, off_bars;   // byte offsets from the 1024-aligned smem base
    // ---- split-K mode (small-M / deep-K layers): CTA u computes K slice u % split of tile u / split ----
    int split, kb_per_split;
    CUtensorMap tmWs;               // fp32 partial tiles in the workspace: [units * 128][block_n]
    float* ws;                      // the same buffer, for the reduction's plain loads
    int* cnt;                       // [2][num_tiles] arrival / departure counters (zero between launches: self-resetting)
    const void* residual;           // raw pointers for the reduction phase
    void* out;
    int ldc, ldr;
};

// one 32-column chunk of this warp's 32 accumulator rows; cb = the warp's smem chunk (holds the residual when RES != 0)
template <bool OUT_F32, int RES, bool GEGLU, bool STATS>
__device__ __forceinline__ void persist_chunk(const PParams& p, uint32_t taddr, int ch, const float* sbv, const float* sbg, uint8_t* cb,
                                              int lane, bool last_chunk, uint64_t* tempty_bar, uint64_t* rfull_bar, uint32_t rparity,
                                              float* gn_dst, int nrows) {
    uint32_t r0[16], r1[16], g0[16], g1[16];
    ptx::tmem_ld_32x32b_x16(taddr + ch * 32, r0);
    ptx::tmem_ld_32x32b_x16(taddr + ch * 32 + 16, r1);
    const int half = p.block_n >> 1;
    if constexpr (GEGLU) {
        ptx::tmem_ld_32x32b_x16(taddr + half + ch * 32, g0);
        ptx::tmem_ld_32x32b_x16(taddr + half + ch * 32 + 16, g1);
    }
    if constexpr (RES != 0) ptx::mbar_wait(rfull_bar, rparity);
    ptx::tmem_ld_wait();
    if (last_chunk) {   // the accumulator stage is free as soon as its last column left TMEM
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(tempty_bar);
    }
    float v[32];
    const float4* sb4 = reinterpret_cast<const float4*>(sbv);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b = sb4[j];   // same address in every lane: broadcast
        const uint32_t* r = j < 4 ? r0 : r1;
        const int o = (j & 3) * 4;
        v[4 * j + 0] = __uint_as_float(r[o + 0]) + b.x;
        v[4 * j + 1] = __uint_as_float(r[o + 1]) + b.y;
        v[4 * j + 2] = __uint_as_float(r[o + 2]) + b.z;
        v[4 * j + 3] = __uint_as_float(r[o + 3]) + b.w;
    }
    if constexpr (GEGLU) {
        const float4* sg4 = reinterpret_cast<const float4*>(sbg);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 b = sg4[j];
            const uint32_t* r = j < 4 ? g0 : g1;
            const int o = (j & 3) * 4;
            v[4 * j + 0] *= gelu_erf_fast(__uint_as_float(r[o + 0]) + b.x);
            v[4 * j + 1] *= gelu_erf_fast(__uint_as_float(r[o + 1]) + b.y);
            v[4 * j + 2] *= gelu_erf_fast(__uint_as_float(r[o + 2]) + b.z);
            v[4 * j + 3] *= gelu_erf_fast(__uint_as_float(r[o + 3]) + b.w);
        }
    }
    // smem chunk layouts = what TMA produces / consumes: fp32 rows of 128 B with the 128-byte swizzle (16-byte piece j of row r
    // at j ^ (r & 7)), bf16 rows of 64 B with the 64-byte swizzle (piece j at j ^ ((r >> 1) & 3))
    uint8_t* row128 = cb + lane * 128;
    uint8_t* row64 = cb + lane * 64;
    const int x128 = lane & 7, x64 = (lane >> 1) & 3;
    if constexpr (RES == 2) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 t = *reinterpret_cast<const float4*>(row128 + ((j ^ x128) << 4));
            v[4 * j + 0] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w;
        }
    } else if constexpr (RES == 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint4 u = *reinterpret_cast<const uint4*>(row64 + ((j ^ x64) << 4));
            float2 f;
            f = unpack_bf16x2(u.x); v[8 * j + 0] += f.x; v[8 * j + 1] += f.y;
            f = unpack_bf16x2(u.y); v[8 * j + 2] += f.x; v[8 * j + 3] += f.y;
            f = unpack_bf16x2(u.z); v[8 * j + 4] += f.x; v[8 * j + 5] += f.y;
            f = unpack_bf16x2(u.w); v[8 * j + 6] += f.x; v[8 * j + 7] += f.y;
        }
    }
    // residual and output rows of different widths overlap across threads: everyone reads before anyone writes
    if constexpr (RES != 0 && ((RES == 2) != OUT_F32)) __syncwarp();
    if constexpr (OUT_F32) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(row128 + ((j ^ x128) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint4 u;
            u.x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
            u.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
            u.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
            u.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
            *reinterpret_cast<uint4*>(row64 + ((j ^ x64) << 4)) = u;
        }
    }
    if constexpr (STATS) {
        // column sums of the finished fp32 chunk: lane c walks column c down the warp's rows (conflict-free: the swizzle
        // permutes 16-byte pieces inside a row, a warp still reads one whole 128-byte row per step)
        __syncwarp();
        float s = 0.f, ss = 0.f;
        const uint8_t* colp = cb + ((lane & 3) << 2);
        const int piece = lane >> 2;
        for (int r = 0; r < nrows; ++r) {
            const float x = *reinterpret_cast<const float*>(colp + r * 128 + ((piece ^ (r & 7)) << 4));
            s += x;
            ss = fmaf(x, x, ss);
        }
        gn_dst[ch * 32 + lane] = s;          // this quarter's slot of the tile's statistics scratch: [sum 256 | sum of squares 256]
        gn_dst[256 + ch * 32 + lane] = ss;
    }
}

template <bool OUT_F32, int RES, bool GEGLU, bool STATS>
__device__ __forceinline__ void persist_epilogue(const PParams& p, uint8_t* smem, uint32_t tmem_base, int warp, int lane) {
    const int ew = warp - 2;  // 0..7
    const int q = warp & 3;   // TMEM lane quarter this warp may access = rows [32q, 32q + 32) of the tile
    const int h = ew >> 2;    // which chunks of the quarter: ch = h, h + 2, ...  (warps 2..5 -> h 0, warps 6..9 -> h 1; quarters distinct in each group)
    const int D = p.depth;
    const int kChunkBytes = p.chunk_bytes;
    uint8_t* my = smem + p.off_epi + (size_t)ew * D * kChunkBytes;
    float* sb = reinterpret_cast<float*>(smem + p.off_bias) + ew * 256;   // [128 value biases | 128 gate biases] of this warp's chunks
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.off_bars);
    uint64_t* tfull = bars + 16;
    uint64_t* tempty = bars + 18;
    uint64_t* rfull = bars + 20 + ew * kMaxDepth;
    const int half = p.block_n >> 1;
    const int nch = (GEGLU ? half : p.block_n) >> 5;
    const int nl = nch > h ? (nch - h + 1) >> 1 : 0;   // chunks of a tile this warp moves
    const int my_tiles = ((int)blockIdx.x < p.num_tiles) ? (p.num_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int total = my_tiles * nl;
    const int out_n = GEGLU ? half : p.block_n;   // output columns per tile

    auto issue_res = [&](int g) {   // lane 0: this warp's g-th residual chunk -> smem chunk g % D
        const int itl = g / nl, ch = h + 2 * (g - itl * nl);
        const int tile = (int)blockIdx.x + itl * (int)gridDim.x;
        const int m_tile = tile / p.n_tiles, n_tile = tile - m_tile * p.n_tiles;
        const int buf = g % D;
        ptx::mbar_expect_tx(&rfull[buf], RES == 2 ? 4096u : 2048u);
        ptx::tma_load_2d(my + buf * kChunkBytes, &p.tmRes, &rfull[buf], n_tile * p.block_n + ch * 32, m_tile * BLOCK_M + q * 32);
    };
    if constexpr (RES != 0) {
        // (holding this prefetch back until the producer's first ring of operand loads is out was measured: the residual then
        // lands too late for a short-K tile -- M8192 N320 K320 7.9 -> 9.0 us -- so it goes out at once)
        if (lane == 0)
            for (int g = 0; g < D && g < total; ++g) issue_res(g);
    }

    int g = 0;
    for (int it = 0; it < my_tiles; ++it) {
        const int tile = (int)blockIdx.x + it * (int)gridDim.x;
        const int m_tile = tile / p.n_tiles, n_tile = tile - m_tile * p.n_tiles;
        const int n0 = n_tile * p.block_n;
        const int row0 = m_tile * BLOCK_M + q * 32;
        // the biases of this warp's chunks (+ the time-embedding row of this warp's image) -> the warp's smem copy
        __syncwarp();
        {
            const int img = p.rowbias ? min(row0, p.M - 1) / p.rows_per_image : 0;
            for (int l = 0; l < nl; ++l) {
                const int c = (h + 2 * l) * 32 + lane;
                float b = p.bias ? __ldg(p.bias + n0 + c) : 0.f;
                if (p.rowbias) b += __ldg(p.rowbias + (size_t)img * p.ldrb + n0 + c);
                sb[l * 32 + lane] = b;
                if constexpr (GEGLU) sb[128 + l * 32 + lane] = p.bias ? __ldg(p.bias + n0 + half + c) : 0.f;
            }
        }
        __syncwarp();
        const int acc = it & 1;
        ptx::mbar_wait(&tfull[acc], (uint32_t)(it >> 1) & 1u);
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t)acc * p.acc_stride + ((uint32_t)(q * 32) << 16);
        const int nrows = max(0, min(32, p.M - row0));
        float* sstat = reinterpret_cast<float*>(smem + p.off_stat);   // [4 quarters][2][256]
        float* gn_dst = STATS ? sstat + q * 512 : nullptr;
        if (nl == 0) {   // nothing to move for this warp (a one-chunk tile): it still takes part in the stage hand-back
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
        }
        for (int l = 0; l < nl; ++l, ++g) {
            const int ch = h + 2 * l;
            const int buf = g % D;
            uint8_t* cb = my + buf * kChunkBytes;
            if constexpr (RES == 0) {
                // the store that last read this chunk (D = 2 chunks ago) must be done with it
                if (lane == 0) ptx::tma_store_wait_read<1>();
                __syncwarp();
            }
            persist_chunk<OUT_F32, RES, GEGLU, STATS>(p, taddr, ch, sb + l * 32, sb + 128 + l * 32, cb, lane, l == nl - 1, &tempty[acc],
                                                     &rfull[buf], (uint32_t)(g / D) & 1u, gn_dst, nrows);
            ptx::fence_proxy_async();   // generic-proxy smem writes -> visible to the TMA (async proxy)
            __syncwarp();
            if (lane == 0) {
                ptx::tma_store_2d(&p.tmOut, cb, n_tile * out_n + ch * 32, row0);
                ptx::tma_store_commit();
                if constexpr (RES != 0) {
                    // chunk g - 1 has been read by its store by now (at most this one still pending): refill it D - 1 ahead
                    if (g >= 1 && g - 1 + D < total) {
                        ptx::tma_store_wait_read<1>();
                        issue_res(g - 1 + D);
                    }
                }
            }
        }
        if constexpr (STATS) {
            // GroupNorm statistics of the tile: the four quarters' column sums folded in a fixed order (bit-reproducible) into
            // ONE partial row per tile, [m_tile][sum | sum of squares][N] -- what b200sd_groupnorm_silu_parts folds per image
            ptx::named_bar_sync(1, kEpiWarps * 32);
            const int te = ew * 32 + lane;
            if (te < p.block_n) {
                float s0 = 0.f, s1 = 0.f;
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) { s0 += sstat[qq * 512 + te]; s1 += sstat[qq * 512 + 256 + te]; }
                float* dst = p.gn_part + (size_t)m_tile * 2 * p.N + n0 + te;
                dst[0] = s0;
                dst[p.N] = s1;
            }
            ptx::named_bar_sync(1, kEpiWarps * 32);   // the scratch is rewritten by the next tile
        }
    }
    if (lane == 0) ptx::tma_store_wait<0>();   // all output writes performed before the CTA may exit
    __syncwarp();
}

// ---- split-K epilogue: K slice s of a tile.  Phase 1: the fp32 partial accumulator goes to the workspace (TMA stores, same
// chunk machinery).  Then the `split` CTAs of the tile meet on an arrival counter in global memory (all CTAs of the grid are
// co-resident: the launch is cooperative and has at most one CTA per SM).  Phase 2: CTA s owns rows [s * 128 / split, ...) of
// the tile: it sums the `split` partials of those rows IN SLICE ORDER (deterministic), adds bias / time embedding / residual,
// stores, and publishes the GroupNorm column statistics of its rows.  The partials never leave L2.
// (The first design exchanged partials over distributed shared memory inside a thread-block cluster: at most 8 slices, clusters
// of 8 placed badly -- 16 of them ran as two waves -- and the pull-style DSMEM reduction took longer than the main loop:
// 10.5 of 22 us on the 8x8 convs.)
template <bool OUT_F32, int RES, bool STATS>
__device__ __forceinline__ void persist_epilogue_split(const PParams& p, uint8_t* smem, uint32_t tmem_base, int warp, int lane) {
    const int ew = warp - 2, q = warp & 3, h = ew >> 2;
    const int kChunkBytes = 4096;
    uint8_t* my = smem + p.off_epi + (size_t)ew * 2 * kChunkBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.off_bars);
    uint64_t* tfull = bars + 16;
    uint64_t* tempty = bars + 18;
    const int unit = blockIdx.x, tile = unit / p.split, s = unit - tile * p.split;
    const int m_tile = tile / p.n_tiles, n_tile = tile - m_tile * p.n_tiles;
    const int n0 = n_tile * p.block_n, m0 = m_tile * BLOCK_M;
    const int nch = p.block_n >> 5;
    const int nl = nch > h ? (nch - h + 1) >> 1 : 0;
    // ---- phase 1: partial accumulator -> workspace ----
    ptx::mbar_wait(&tfull[0], 0);
    ptx::tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
    for (int l = 0; l < nl; ++l) {
        const int ch = h + 2 * l;
        uint8_t* cb = my + (l & 1) * kChunkBytes;
        if (lane == 0) ptx::tma_store_wait_read<1>();
        __syncwarp();
        uint32_t r0[16], r1[16];
        ptx::tmem_ld_32x32b_x16(taddr + ch * 32, r0);
        ptx::tmem_ld_32x32b_x16(taddr + ch * 32 + 16, r1);
        ptx::tmem_ld_wait();
        uint8_t* row128 = cb + lane * 128;
        const int x128 = lane & 7;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t* r = j < 4 ? r0 : r1;
            const int o = (j & 3) * 4;
            *reinterpret_cast<uint4*>(row128 + ((j ^ x128) << 4)) = make_uint4(r[o], r[o + 1], r[o + 2], r[o + 3]);
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            ptx::tma_store_2d(&p.tmWs, cb, ch * 32, unit * BLOCK_M + q * 32);
            ptx::tma_store_commit();
        }
    }
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) {
        ptx::mbar_arrive(&tempty[0]);
        ptx::tma_store_wait<0>();        // this warp's partial rows are written
        ptx::fence_proxy_async_global(); // async-proxy writes -> ordered before the generic-proxy release below
        __threadfence();
    }
    ptx::named_bar_sync(1, kEpiWarps * 32);
    const int te = ew * 32 + lane;
    int* cnt_in = p.cnt + tile;
    int* cnt_out = p.cnt + p.num_tiles + tile;
    if (te == 0) {
        atomicAdd(cnt_in, 1);
        int seen;
        long long t0 = clock64();
        do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(cnt_in) : "memory");
            if (clock64() - t0 > 4000000000LL) { printf("b200sd: split-K arrival wait timed out (unit %d)\n", unit); __trap(); }
        } while (seen < p.split);
        __threadfence();
    }
    ptx::named_bar_sync(1, kEpiWarps * 32);
    // ---- phase 2: rows [s * rpc, (s + 1) * rpc) of the tile, all block_n columns ----
    const int rpc = BLOCK_M / p.split;
    const int groups = p.block_n >> 2;                 // float4 column groups
    const int rslots = (kEpiWarps * 32) / groups < 4 ? (kEpiWarps * 32) / groups : 4;
    const int c4 = te % groups, rslot = te / groups;
    float* sstat = reinterpret_cast<float*>(smem + p.off_stat);   // [4][2][256]
    float cs[4] = {0.f, 0.f, 0.f, 0.f}, cq[4] = {0.f, 0.f, 0.f, 0.f};
    if (rslot < rslots) {
        const int col = n0 + c4 * 4;
        float4 b4 = p.bias ? __ldg(reinterpret_cast<const float4*>(p.bias + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = rslot; r < rpc; r += rslots) {
            const int trow = s * rpc + r;                // row inside the tile
            const int grow = m0 + trow;
            if (grow >= p.M) break;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const float* src = p.ws + ((size_t)(tile * p.split) * BLOCK_M + trow) * p.block_n + c4 * 4;
            for (int j = 0; j < p.split; ++j) {
                const float4 t = __ldcg(reinterpret_cast<const float4*>(src + (size_t)j * BLOCK_M * p.block_n));
                v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
            }
            v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
            if (p.rowbias) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(p.rowbias + (size_t)(grow / p.rows_per_image) * p.ldrb + col));
                v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
            }
            if constexpr (RES == 2) {
                const float4 t = __ldcg(reinterpret_cast<const float4*>(static_cast<const float*>(p.residual) + (size_t)grow * p.ldr + col));
                v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
            } else if constexpr (RES == 1) {
                const uint2 u = __ldcg(reinterpret_cast<const uint2*>(static_cast<const bf16*>(p.residual) + (size_t)grow * p.ldr + col));
                const float2 f0 = unpack_bf16x2(u.x), f1 = unpack_bf16x2(u.y);
                v.x += f0.x; v.y += f0.y; v.z += f1.x; v.w += f1.y;
            }
            if constexpr (STATS) {
                cs[0] += v.x; cs[1] += v.y; cs[2] += v.z; cs[3] += v.w;
                cq[0] = fmaf(v.x, v.x, cq[0]); cq[1] = fmaf(v.y, v.y, cq[1]); cq[2] = fmaf(v.z, v.z, cq[2]); cq[3] = fmaf(v.w, v.w, cq[3]);
            }
            if constexpr (OUT_F32) {
                *reinterpret_cast<float4*>(static_cast<float*>(p.out) + (size_t)grow * p.ldc + col) = v;
            } else {
                uint2 u;
                u.x = pack_bf16x2(v.x, v.y);
                u.y = pack_bf16x2(v.z, v.w);
                *reinterpret_cast<uint2*>(static_cast<bf16*>(p.out) + (size_t)grow * p.ldc + col) = u;
            }
        }
    }
    if constexpr (STATS) {
        // column statistics of this CTA's rows: the row slots folded in a fixed order; partial row = m_tile * split + s (the
        // n-tiles of a row band write disjoint column ranges of the same partial row)
        if (rslot < 4) {
#pragma unroll
            for (int i = 0; i < 4; ++i) { sstat[rslot * 512 + c4 * 4 + i] = cs[i]; sstat[rslot * 512 + 256 + c4 * 4 + i] = cq[i]; }
        }
        ptx::named_bar_sync(1, kEpiWarps * 32);
        if (te < p.block_n) {
            float s0 = 0.f, s1 = 0.f;
            for (int rs = 0; rs < rslots; ++rs) { s0 += sstat[rs * 512 + te]; s1 += sstat[rs * 512 + 256 + te]; }
            float* dst = p.gn_part + (size_t)(m_tile * p.split + s) * 2 * p.N + n0 + te;
            dst[0] = s0;
            dst[p.N] = s1;
        }
    }
    // ---- departure: the last CTA of the tile to finish reading re-arms both counters for the next launch ----
    ptx::named_bar_sync(1, kEpiWarps * 32);
    if (te == 0) {
        __threadfence();
        if (atomicAdd(cnt_out, 1) == p.split - 1) {
            *cnt_out = 0;
            *cnt_in = 0;
            __threadfence();
        }
    }
}

__global__ void __launch_bounds__(kPersistThreads, 1) gemm_persist_kernel(const __grid_constant__ PParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + p.off_b;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.off_bars);
    uint64_t* full_bar = bars;            // [8]
    uint64_t* empty_bar = bars + 8;       // [8]
    uint64_t* tfull = bars + 16;          // [2]  accumulator stage ready for the epilogue
    uint64_t* tempty = bars + 18;         // [2]  accumulator stage drained (one arrival per epilogue warp)
    uint64_t* rfull = bars + 20;          // [8 warps][3]  residual chunk landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20 + kEpiWarps * kMaxDepth);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int b_bytes = p.block_n * BLOCK_K * 2;

    // ---- TMA producers, resumable.  TWO threads feed the ring: thread 0 loads the A tiles, lane 0 of the last warp the B
    // (weight) tiles -- issuing a cp.async.bulk.tensor costs the issuing thread a few hundred cycles, and with both loads of a
    // k-block on one thread that thread, not the memory system, paced the main loop of a one-CTA-per-SM grid (measured: adding
    // ~300 cycles of index arithmetic per k-block to the single producer slowed an M8192 K2880 conv from 22.6 to 33.1 us).
    // All per-tile index arithmetic is hoisted out of the k loop; the first ring of loads is issued BEFORE the CTA-wide prologue
    // sync, so the load latency of the first tile overlaps the TMEM allocation and the barrier hand-shake. ----
    const bool splitk = p.split > 1;
    // work items: whole tiles blockIdx.x, blockIdx.x + gridDim.x, ... -- or, in split-K mode, ONE K slice of one tile
    const int sk_tile = splitk ? (int)blockIdx.x / p.split : 0, sk_s = splitk ? (int)blockIdx.x - sk_tile * p.split : 0;
    // slice s = k-blocks [s * nkb / split, (s + 1) * nkb / split): never empty while nkb >= split
    const int sk_kb0 = splitk ? (sk_s * p.num_k_blocks) / p.split : 0;
    const int sk_kb1 = splitk ? ((sk_s + 1) * p.num_k_blocks) / p.split : p.num_k_blocks;
    int pr_stage = 0, pr_tile = splitk ? sk_tile : (int)blockIdx.x, pr_kb = sk_kb0, pr_m0 = 0, pr_n0 = 0, pr_img = 0, pr_y0 = 0, pr_x0 = 0, pr_tap = 0,
        pr_cb = 0;
    bool pr_new = true;
    uint32_t pr_phase = 0;
    // what: bit 0 = issue the A load, bit 1 = issue the B load, 0 = only advance the cursor (the B producer skips the first ring,
    // which thread 0 issued in full before the prologue sync)
    auto produce = [&](int limit, const int what) {
        const bool load_a = what & 1, load_b = what & 2;
        while (limit > 0 && pr_tile < p.num_tiles) {
            if (pr_new) {   // new work item
                pr_new = false;
                const int m_tile = pr_tile / p.n_tiles, n_tile = pr_tile - m_tile * p.n_tiles;
                pr_m0 = m_tile * BLOCK_M;
                pr_n0 = n_tile * p.block_n;
                if (p.conv) {
                    if (p.tile_n > 1) { pr_img = m_tile * p.tile_n; pr_y0 = 0; }
                    else {
                        int mt = m_tile;
                        if (p.tiles_x > 1) { pr_x0 = (mt % p.tiles_x) * p.tile_w; mt /= p.tiles_x; }
                        pr_img = mt / p.tiles_y; pr_y0 = (mt - pr_img * p.tiles_y) * p.tile_h;
                    }
                }
                pr_tap = pr_kb / p.cblocks;           // 0 unless this is a K slice
                pr_cb = pr_kb - pr_tap * p.cblocks;
            }
            uint64_t* fb = &full_bar[pr_stage];
            if (what) ptx::mbar_wait(&empty_bar[pr_stage], pr_phase ^ 1);
            if (load_a) {
                ptx::mbar_expect_tx(fb, (uint32_t)kABytes);      // full barriers count two arrivals: one per operand

                uint8_t* dst_a = smem_a + (size_t)pr_stage * kABytes;
                if (!p.conv) {
                    if (pr_kb < p.cblocks0) ptx::tma_load_2d(dst_a, &p.tmA0, fb, pr_kb * BLOCK_K, pr_m0);
                    else ptx::tma_load_2d(dst_a, &p.tmA1, fb, (pr_kb - p.cblocks0) * BLOCK_K, pr_m0);
                } else {
                    const int dy = pr_tap / 3 - 1, dx = pr_tap - (pr_tap / 3) * 3 - 1;
                    if (pr_cb < p.cblocks0) ptx::tma_load_4d(dst_a, &p.tmA0, fb, pr_cb * BLOCK_K, pr_x0 + dx, pr_y0 + dy, pr_img);
                    else ptx::tma_load_4d(dst_a, &p.tmA1, fb, (pr_cb - p.cblocks0) * BLOCK_K, pr_x0 + dx, pr_y0 + dy, pr_img);
                }
            }
            if (load_b) {
                ptx::mbar_expect_tx(fb, (uint32_t)b_bytes);
                ptx::tma_load_2d(smem_b + (size_t)pr_stage * b_bytes, &p.tmB, fb, pr_kb * BLOCK_K, pr_n0);
            }
            if (++pr_stage == p.stages) { pr_stage = 0; pr_phase ^= 1; }
            if (++pr_cb == p.cblocks) { pr_cb = 0; ++pr_tap; }
            if (++pr_kb == sk_kb1) { pr_kb = 0; pr_new = true; pr_tile = splitk ? p.num_tiles : pr_tile + (int)gridDim.x; }
            --limit;
        }
    };
    const bool is_prod_a = threadIdx.x == 0, is_prod_b = threadIdx.x == kPersistThreads - 32;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&p.tmA0);
        ptx::prefetch_tmap(&p.tmB);
        ptx::prefetch_tmap(&p.tmOut);
        if (p.cblocks0 != p.cblocks) ptx::prefetch_tmap(&p.tmA1);
        if (p.res_kind) ptx::prefetch_tmap(&p.tmRes);
        for (int s = 0; s < p.stages; ++s) {
            ptx::mbar_init(&full_bar[s], 2);     // A producer + B producer
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(&tfull[s], 1);
            ptx::mbar_init(&tempty[s], kEpiWarps);
        }
        for (int s = 0; s < kEpiWarps * kMaxDepth; ++s) ptx::mbar_init(&rfull[s], 1);
        ptx::fence_barrier_init();
        produce(p.stages, 3);     // first ring, both operands; every ring slot is free: none of these waits blocks
    }
    if (warp == 1) {
        ptx::tmem_alloc(tmem_slot, p.tmem_cols);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer of the A tiles (its first ring of loads went out before the CTA-wide sync above) =================
        if (is_prod_a) produce(0x7fffffff, 1);
    } else if (warp == kPersistThreads / 32 - 1) {
        // ================= TMA producer of the B (weight) tiles =================
        if (is_prod_b) {
            produce(p.stages, 0);      // thread 0 issued the first ring
            produce(0x7fffffff, 2);
        }
    } else if (warp == 1) {
        // ================= MMA issuer (one elected thread) =================
        if (ptx::elect_one()) {
            const uint32_t idesc = ptx::umma_idesc_bf16(BLOCK_M, (uint32_t)p.block_n);
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            const int nkb = sk_kb1 - sk_kb0;      // k-blocks per work item
            for (int tile = splitk ? sk_tile : (int)blockIdx.x; tile < p.num_tiles; tile = splitk ? p.num_tiles : tile + (int)gridDim.x, ++it) {
                const int acc = it & 1;
                ptx::mbar_wait(&tempty[acc], ((uint32_t)(it >> 1) & 1u) ^ 1u);   // the epilogue has drained this stage
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)acc * p.acc_stride;
                for (int kb = 0; kb < nkb; ++kb) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint64_t da = ptx::umma_desc_k_sw128(ptx::smem_u32(smem_a + (size_t)stage * kABytes));
                    const uint64_t db = ptx::umma_desc_k_sw128(ptx::smem_u32(smem_b + (size_t)stage * b_bytes));
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                        ptx::umma_bf16_ss(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
                    ptx::umma_commit(&empty_bar[stage]);   // frees the smem slot when these MMAs retire
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
                ptx::umma_commit(&tfull[acc]);
            }
        }
    } else {
        // ================= epilogue warps =================
        const int variant = (p.geglu ? 100 : 0) + (p.out_f32 ? 10 : 0) + p.res_kind + (p.gn_part ? 1000 : 0);
        if (splitk) {
            switch (variant) {
                case 0: persist_epilogue_split<false, 0, false>(p, smem, tmem_base, warp, lane); break;
                case 1: persist_epilogue_split<false, 1, false>(p, smem, tmem_base, warp, lane); break;
                case 2: persist_epilogue_split<false, 2, false>(p, smem, tmem_base, warp, lane); break;
                case 10: persist_epilogue_split<true, 0, false>(p, smem, tmem_base, warp, lane); break;
                case 11: persist_epilogue_split<true, 1, false>(p, smem, tmem_base, warp, lane); break;
                case 12: persist_epilogue_split<true, 2, false>(p, smem, tmem_base, warp, lane); break;
                case 1010: persist_epilogue_split<true, 0, true>(p, smem, tmem_base, warp, lane); break;
                case 1012: persist_epilogue_split<true, 2, true>(p, smem, tmem_base, warp, lane); break;
                default: break;
            }
        } else
        switch (variant) {
            case 100: persist_epilogue<false, 0, true, false>(p, smem, tmem_base, warp, lane); break;
            case 0: persist_epilogue<false, 0, false, false>(p, smem, tmem_base, warp, lane); break;
            case 1: persist_epilogue<false, 1, false, false>(p, smem, tmem_base, warp, lane); break;
            case 2: persist_epilogue<false, 2, false, false>(p, smem, tmem_base, warp, lane); break;
            case 10: persist_epilogue<true, 0, false, false>(p, smem, tmem_base, warp, lane); break;
            case 11: persist_epilogue<true, 1, false, false>(p, smem, tmem_base, warp, lane); break;
            case 12: persist_epilogue<true, 2, false, false>(p, smem, tmem_base, warp, lane); break;
            case 1010: persist_epilogue<true, 0, false, true>(p, smem, tmem_base, warp, lane); break;
            case 1012: persist_epilogue<true, 2, false, true>(p, smem, tmem_base, warp, lane); break;
            default: break;   // the host never launches another combination
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, p.tmem_cols);
    }
}

uint32_t pow2_cols(int n) {
    uint32_t c = 32;
    while ((int)c < n) c <<= 1;
    return c;
}

int pick_block_n(int N, int m_tiles, int epilogue, bool can_split = false) {
    // Legal tile widths: multiple of 16 (32 for GEGLU), <= 256, dividing N.  Prefer 160 (two CTAs per SM,
    // 90 % of the smem read bandwidth the MMA needs); when that leaves the machine more than half empty
    // (small-M layers) fall to a narrower tile so more CTAs stream operands concurrently.
    const int step = (epilogue == B200SD_EPI_GEGLU) ? 32 : 16;
    const int sms = b200sd_num_sms();
    int best = 0;
    for (int bn = 160; bn >= 64; bn -= step)
        if (N % bn == 0) { best = bn; break; }
    if (best == 0) {
        for (int bn = 256; bn >= step; bn -= step)
            if (N % bn == 0) { best = bn; break; }
        return best;
    }
    // Deep-K layers fill the machine with split-K clusters instead (measured, tools/conv_small_check.py: a 160-wide tile split
    // 4-8 ways beats an 80-wide tile by 25-40 % on the M = 128 ... 2048 convs); only short-K layers narrow their tiles.
    if (epilogue == B200SD_EPI_LINEAR && !can_split && (long)m_tiles * (N / best) * 2 <= sms) {
        for (int bn = 80; bn < best; bn += step)  // narrowest tile (>= 80) that still fits one wave
            if (N % bn == 0 && (long)m_tiles * (N / bn) <= sms) { best = bn; break; }
    }
    return best;
}


// Shared tail of every entry point: pipeline depth, smem budget, launch.
// Grids that fit in one wave keep every k-block of a short K loop in flight (deep ring, 1 CTA/SM);
// larger grids stay <= ~110 KB so two CTAs share an SM and overlap epilogue with main loop.
typedef void (*gemm_kernel_t)(const KParams);
gemm_kernel_t gemm_entry(int pair, int op) {
    switch ((op << 1) | (pair ? 1 : 0)) {
        case 0: return gemm_tcgen05_kernel<false, 0>;
        case 1: return gemm_tcgen05_kernel<true, 0>;
        case 2: return gemm_tcgen05_kernel<false, 1>;
        case 3: return gemm_tcgen05_kernel<true, 1>;
        case 4: return gemm_tcgen05_kernel<false, 2>;
        case 5: return gemm_tcgen05_kernel<true, 2>;
        case 6: return gemm_tcgen05_kernel<false, 3>;
        default: return gemm_tcgen05_kernel<true, 3>;
    }
}

// The opt-in to > 48 KB of dynamic smem is a per-DEVICE function attribute: configure every kernel once per device
// (a second GPU in the same process would otherwise launch without it), under a mutex (the C ABI may be called from threads).
int configure_gemm_kernels() {
    static std::mutex mu;
    static bool configured[64] = {};
    int dev = 0;
    B200SD_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (dev < 0 || dev >= 64 || configured[dev]) return B200SD_OK;
    for (int i = 0; i < 8; ++i) {
        B200SD_CUDA(cudaFuncSetAttribute(gemm_entry(i & 1, i >> 1), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024)));
        B200SD_CUDA(cudaFuncSetAttribute(gemm_entry(i & 1, i >> 1), cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    }
    B200SD_CUDA(cudaFuncSetAttribute(gemm_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024)));
    B200SD_CUDA(cudaFuncSetAttribute(gemm_persist_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    configured[dev] = true;
    return B200SD_OK;
}

// ---- persistent path (gemm_persist_kernel): tile width, eligibility, launch ----
bool persist_enabled() { return g_persist != 0; }
// Tile width for the persistent kernel: a multiple of 32 (its epilogue chunk; 64 for GEGLU: values | gates) dividing N.
// cost = rounds of tiles per SM x operand bytes a tile pulls per k-block (128 + bn rows): the smallest tile that still
// fits one round wins on short grids (more CTAs, shorter epilogue), wide tiles win once several rounds are needed anyway.
int pick_block_n_persist(int N, int m_tiles, bool geglu) {
    const int sms = b200sd_num_sms();
    const int step = geglu ? 64 : 32;
    long best_cost = 0;
    int best = 0;
    for (int bn = step; bn <= 256; bn += step) {
        if (N % bn) continue;
        const long tiles = (long)m_tiles * (N / bn);
        const long cost = ((tiles + sms - 1) / sms) * (BLOCK_M + bn);
        if (best == 0 || cost < best_cost || (cost == best_cost && bn > best)) { best = bn; best_cost = cost; }
    }
    return best;
}

int launch_persist(const b200sd_gemm_args* a, const KParams& k, int m_tiles, b200sd_stream_t stream) {
    PParams p;
    memset(&p, 0, sizeof(p));
    p.tmA0 = k.tmA0; p.tmA1 = k.tmA1; p.tmB = k.tmB;
    p.bias = k.bias; p.rowbias = k.rowbias; p.gn_part = k.gn_part;
    p.M = k.M; p.N = k.N;
    p.num_k_blocks = k.num_k_blocks; p.block_n = k.block_n;
    p.conv = k.conv; p.cblocks0 = k.cblocks0; p.cblocks = k.cblocks;
    p.tile_h = k.tile_h; p.tile_n = k.tile_n; p.tiles_y = k.tiles_y;
    p.tile_w = k.tile_w; p.tiles_x = k.tiles_x;
    p.n_tiles = k.N / k.block_n;
    p.num_tiles = m_tiles * p.n_tiles;
    p.ldrb = k.ldrb; p.rows_per_image = k.rows_per_image;
    p.geglu = k.epilogue == B200SD_EPI_GEGLU;
    p.out_f32 = k.out_f32;
    p.res_kind = k.residual ? (k.res_f32 ? 2 : 1) : 0;
    p.depth = p.res_kind ? kMaxDepth : 2;
    p.split = k.psplit > 1 ? k.psplit : 1;
    p.kb_per_split = ceil_div(k.num_k_blocks, p.split);
    p.residual = k.residual; p.out = k.out; p.ldc = k.ldc; p.ldr = k.ldr;
    const int units = p.num_tiles * p.split;
    if (p.split > 1) {
        B200SD_REQUIRE(k.num_k_blocks >= p.split, "gemm(split-K): fewer K blocks (%d) than slices (%d)", k.num_k_blocks, p.split);
        B200SD_REQUIRE(units <= b200sd_num_sms() && (size_t)units * BLOCK_M * k.block_n * sizeof(float) <= kWsPartialBytes &&
                           (size_t)2 * p.num_tiles * sizeof(int) <= kWsCounterBytes,
                       "gemm(split-K): %d units do not fit the workspace / the machine", units);
        p.depth = 2;     // no residual prefetch: the residual is read in the reduction phase
        p.ws = static_cast<float*>(a->workspace);
        p.cnt = reinterpret_cast<int*>(static_cast<char*>(a->workspace) + kWsPartialBytes);
        const uint64_t dims[2] = {(uint64_t)k.block_n, (uint64_t)units * BLOCK_M};
        const uint64_t str[2] = {0, (uint64_t)k.block_n * 4};
        const uint32_t box[2] = {32, 32};
        const int rc = b200sd_make_tmap(&p.tmWs, a->workspace, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
        if (rc) return rc;
    }
    const int bn = k.block_n;
    p.acc_stride = bn <= 128 ? 128 : 256;
    p.tmem_cols = 2 * p.acc_stride;
    // ---- output / residual tensor maps: 32-column x 32-row boxes (one epilogue chunk of one warp) ----
    const int out_cols = p.geglu ? k.N / 2 : k.N;
    {
        const uint64_t dims[2] = {(uint64_t)out_cols, (uint64_t)k.M};
        const uint64_t str[2] = {0, (uint64_t)k.ldc * (k.out_f32 ? 4 : 2)};
        const uint32_t box[2] = {32, 32};
        const int rc = b200sd_make_tmap(&p.tmOut, k.out, 2, dims, str, box, k.out_f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                                        k.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
        if (rc) return rc;
    }
    if (p.res_kind) {
        const uint64_t dims[2] = {(uint64_t)k.N, (uint64_t)k.M};
        const uint64_t str[2] = {0, (uint64_t)k.ldr * (k.res_f32 ? 4 : 2)};
        const uint32_t box[2] = {32, 32};
        const int rc = b200sd_make_tmap(&p.tmRes, k.residual, 2, dims, str, box, k.res_f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                                        k.res_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
        if (rc) return rc;
    }
    // ---- smem layout ----
    const int stage_bytes = kABytes + bn * BLOCK_K * 2;
    p.chunk_bytes = (p.out_f32 || p.res_kind == 2 || k.psplit > 1) ? 4096 : 2048;
    const int epi_bytes = kEpiWarps * p.depth * p.chunk_bytes;
    const int bias_bytes = kEpiWarps * 256 * (int)sizeof(float);
    const int stat_bytes = k.gn_part ? 4 * 2 * 256 * (int)sizeof(float) : 0;
    const int bars_bytes = 512;
    const int budget = 227 * 1024 - 1024;
    int stages = (budget - epi_bytes - bias_bytes - stat_bytes - bars_bytes) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    B200SD_REQUIRE(stages >= 2, "gemm(persistent): smem budget leaves %d stages for block_n %d", stages, bn);
    p.stages = stages;
    p.off_b = (uint32_t)stages * kABytes;
    p.off_epi = (uint32_t)stages * stage_bytes;
    p.off_bias = p.off_epi + epi_bytes;
    p.off_stat = p.off_bias + bias_bytes;
    p.off_bars = p.off_stat + stat_bytes;
    const size_t smem_bytes = (size_t)p.off_bars + bars_bytes + 1024;
    {
        const int rc = configure_gemm_kernels();
        if (rc) return rc;
    }
    const int sms = b200sd_num_sms();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.split > 1 ? units : (p.num_tiles < sms ? p.num_tiles : sms));
    cfg.blockDim = dim3(kPersistThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    if (p.split > 1) {   // the K slices of a tile wait for one another: every CTA of the grid must be resident
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    B200SD_CUDA(cudaLaunchKernelEx(&cfg, gemm_persist_kernel, p));
    g_b200sd_launches.fetch_add(1, std::memory_order_relaxed);
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

int launch_gemm(KParams& p, int m_tiles, int n_tiles, int grid_z, bool cluster, b200sd_stream_t stream) {
    const int sms = b200sd_num_sms();
    const int bn = p.block_n;
    if (p.pair) m_tiles = (m_tiles + 1) & ~1;   // an odd tail gets a dummy peer (TMA zero-fills, the epilogue stores nothing)
    const int stage_bytes = kABytes + ((bn * BLOCK_K * 2) >> (p.pair ? 1 : 0));
    const long total_ctas = (long)m_tiles * n_tiles * grid_z;
    int stages;
    if (total_ctas <= sms || bn > 160) stages = (200 * 1024) / stage_bytes;
    else stages = (108 * 1024) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages > p.kb_per_split && total_ctas <= sms) stages = p.kb_per_split;
    const int min_stages = ceil_div(BLOCK_M * (bn + 4) * (int)sizeof(float), stage_bytes);  // epilogue staging tile
    if (stages < min_stages) stages = min_stages;
    if (stages < 2) stages = 2;
    p.stages = stages;
    B200SD_REQUIRE((size_t)stages * stage_bytes >= (size_t)BLOCK_M * (bn + 4) * sizeof(float), "gemm: smem ring smaller than the epilogue staging tile");
    const size_t smem_bytes = (size_t)stages * stage_bytes + 1024 /*align slack*/ + 256 /*barriers*/ + 3072 /*bias tiles*/;
    B200SD_REQUIRE(smem_bytes <= 227 * 1024, "gemm: smem budget exceeded (%zu B)", smem_bytes);

    {
        const int rc = configure_gemm_kernels();
        if (rc) return rc;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(m_tiles, n_tiles, grid_z);
    cfg.blockDim = dim3(kNumThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    if ((cluster && grid_z > 1) || p.pair) {
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = p.pair ? 2 : 1;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = p.pair ? 1 : grid_z;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    B200SD_CUDA(cudaLaunchKernelEx(&cfg, gemm_entry(p.pair, p.b_mode), p));
    g_b200sd_launches.fetch_add(1, std::memory_order_relaxed);
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// CTA pairs (cta_group::2): 0 = auto, 1 = force, -1 = off
// Measured on B200 (tools/pair_check.py): pairs win 5-13 % on long-K tiles of grids that fill the machine
// (conv3x3 at batch 8: 1171 -> 1325 TFLOP/s) and lose ~5 % on short-K GEMMs (one more cluster barrier per tile).
bool want_pair(int request, int split, int m_tiles, int n_tiles, int k_blocks) {
    if (request < 0 || split != 1) return false;
    if (request > 0) return true;
    return m_tiles >= 2 && k_blocks >= 32 && (long)m_tiles * n_tiles >= b200sd_num_sms();
}

// Tile width for MN-major B operands (64-column TMA boxes), from the sweep in tools/bwd_gemm_bench.py (B200, batch 8):
// 128 wins or ties for dgrad (plain and conv) and conv wgrad (two CTAs per SM survive: 3 x 32 KB stages + the staging tile);
// 192 for plain wgrad (long K, small output).  64 is never better than 128 when N > 64.  Wider tiles were re-measured after the
// kernel learnt to load only the live boxes of a narrow last tile: still slower (one CTA per SM).
// kind: 0 dgrad, 1 wgrad plain, 2 wgrad conv.
int pick_block_n_mn(int N, int m_tiles, int kind) {
    int best;
    if (N <= 64) best = 64;
    else if (N <= 128) best = 128;
    else if (kind == 1) best = N <= 192 ? 192 : ((N % 192 == 0 || N % 128 != 0) ? 192 : (N % 256 == 0 ? 256 : 128));
    else best = (N % 192 == 0 && N % 128 != 0) ? 192 : 128;
    // small grids: narrower tiles put more CTAs in flight
    while (best > 64 && (long)m_tiles * ceil_div(N, best) * 2 <= b200sd_num_sms()) best -= 64;
    return best;
}

// conv geometry shared by forward / dgrad: M tile = (tile_w x tile_h x tile_n) pixels <= 128
int conv_m_tiling(KParams& p, int NB, int H, int W, int M, int* m_tiles) {
    B200SD_REQUIRE(NB > 0 && H > 0 && W > 0 && M == NB * H * W, "gemm(conv): M=%d != batch*H*W", M);
    p.tiles_x = 1;
    if (W > BLOCK_M) {
        // an image row is wider than one tile (VAE at 256 / 512 pixels): a tile = 128 consecutive pixels of ONE row, box
        // (64 ch, 128, 1, 1) at x0 = tile_x * 128; the halo columns x0 - 1 / x0 + 128 come from the neighbouring pixels of the
        // same row (or TMA zero fill at the image border), exactly as for whole-row tiles
        B200SD_REQUIRE(W % BLOCK_M == 0, "gemm(conv): W=%d > 128 must be a multiple of 128", W);
        p.tile_w = BLOCK_M; p.tile_h = 1; p.tile_n = 1;
        p.tiles_x = W / BLOCK_M; p.tiles_y = H;
        p.rows_valid = BLOCK_M;
        p.a_bytes = p.rows_valid * BLOCK_K * 2;
        *m_tiles = NB * H * p.tiles_x;
        return B200SD_OK;
    }
    const int max_h = BLOCK_M / W;
    if (H <= max_h) {
        p.tile_h = H;
        p.tile_n = max_h / H;
        if (p.tile_n < 1) p.tile_n = 1;
        if (p.tile_n > NB) p.tile_n = NB;
    } else {
        p.tile_n = 1;
        p.tile_h = 1;
        for (int h = max_h; h >= 1; --h)
            if (H % h == 0) { p.tile_h = h; break; }
    }
    p.tile_w = W;
    p.tiles_y = H / p.tile_h;
    p.rows_valid = p.tile_w * p.tile_h * p.tile_n;
    p.a_bytes = p.rows_valid * BLOCK_K * 2;
    *m_tiles = (p.tile_n > 1) ? ceil_div(NB, p.tile_n) : NB * p.tiles_y;
    return B200SD_OK;
}

}  // namespace

// Split-K scratch of the persistent kernel: fp32 partial tiles (at most one 128 x 256 tile per SM) + the per-tile counters.
// The counters must be ZERO before the first launch that uses the buffer (the kernel leaves them zeroed).
extern "C" size_t b200sd_gemm_workspace_bytes(void) { return kWsPartialBytes + kWsCounterBytes; }

extern "C" int b200sd_geglu_tile(int N) {
    // the persistent kernel moves 32-column chunks of values and gates: tile = [tile/2 values | tile/2 gates], tile % 64 == 0
    // ... except for the widest feed-forward (N = 8C = 10240, only ever run at M <= 512 rows at 64x64 latents): 160 tiles of 256
    // columns on 148 SMs would leave a second, nearly empty round; it keeps the 160-wide tiles of gemm_tcgen05_kernel (measured
    // with cold weights: 19.2 us vs 24.9 persistent)
    if (persist_enabled() && N < 10240) {
        if (N % 256 == 0) return 256;
        if (N % 128 == 0) return 128;
        if (N % 64 == 0) return 64;
    }
    return pick_block_n(N, 1, B200SD_EPI_GEGLU);
}

// M / N / split-K tiling of a forward GEMM (shared by the launch and by b200sd_gemm_gn_layout, which tells the consumer of
// the GroupNorm column statistics how many partial rows each image owns).  Fills the tiling fields of p.
static int gemm_tiling(const b200sd_gemm_args* a, KParams& p, int* m_tiles_out, int* n_tiles_out) {
    const int C0 = a->C0, C1 = a->a1 ? a->C1 : 0, C = C0 + C1;
    (void)C;
    // ---- M tiling ----
    if (!p.conv) {
        p.rows_valid = BLOCK_M;
        p.a_bytes = kABytes;
        p.tile_w = p.tile_h = p.tile_n = 1;
        p.tiles_x = 1;
        p.tiles_y = 1;
        *m_tiles_out = ceil_div(a->M, BLOCK_M);
    } else {
        const int rc = conv_m_tiling(p, a->batch, a->H, a->W, a->M, m_tiles_out);
        if (rc) return rc;
    }

    const int m_tiles = *m_tiles_out;

    // ---- N tiling ----
    const bool can_split = a->split_k <= 0 && a->epilogue == B200SD_EPI_LINEAR && p.num_k_blocks >= 16;
    int bn = a->block_n > 0 ? a->block_n : pick_block_n(a->N, m_tiles, a->epilogue, can_split);
    B200SD_REQUIRE(bn >= 16 && bn <= 256 && bn % 16 == 0 && a->N % bn == 0, "gemm: bad block_n %d for N=%d", bn, a->N);
    B200SD_REQUIRE(a->epilogue != B200SD_EPI_GEGLU || bn % 32 == 0, "gemm: GEGLU needs block_n %% 32 == 0");
    p.block_n = bn;
    int n_tiles = a->N / bn;
    p.tmem_cols = pow2_cols(bn);

    // ---- split-K: the splits of a tile form a thread-block cluster (<= 8 CTAs) and reduce over DSMEM ----
    const int sms = b200sd_num_sms();
    int split = a->split_k;
    if (split <= 0) {
        split = 1;
        const int tiles = m_tiles * n_tiles;
        if (a->epilogue == B200SD_EPI_LINEAR && tiles * 2 <= sms && p.num_k_blocks >= 16) {
            while (split < 8 && tiles * split * 2 <= sms && p.num_k_blocks / (split * 2) >= 8) split *= 2;
        }
    }
    int n_tiles_f = n_tiles;
    if (a->split_k <= 0 && a->block_n <= 0 && can_split) {
        // clusters of 8 only place well up to ~8 of them (measured: 16 clusters of 8 run as two waves); and when the split
        // grid still leaves half the machine idle, halve the tile width instead of splitting deeper
        const int tiles = m_tiles * n_tiles;
        if (split == 8 && tiles > 8) split = 4;
        if (split <= 4 && tiles * split * 2 <= sms && bn % 32 == 0 && bn / 2 >= 80) {
            bn /= 2;
            p.block_n = bn;
            n_tiles_f = a->N / bn;
            p.tmem_cols = pow2_cols(bn);
        }
    }
    B200SD_REQUIRE(split == 1 || a->epilogue == B200SD_EPI_LINEAR, "gemm: split-K only with the linear epilogue");
    B200SD_REQUIRE(split == 1 || split == 2 || split == 4 || split == 8, "gemm: split_k must be 1, 2, 4 or 8 (cluster size)");
    p.kb_per_split = ceil_div(p.num_k_blocks, split);
    B200SD_REQUIRE((split - 1) * p.kb_per_split < p.num_k_blocks, "gemm: split_k=%d leaves an empty split for K=%d", split, a->K);
    *n_tiles_out = n_tiles_f;
    p.split_k = split;
    p.pair = want_pair(a->pair, split, m_tiles, n_tiles_f, p.num_k_blocks) && bn % 32 == 0;
    // ---- persistent kernel (TMA-store epilogue, double-buffered TMEM): un-split, un-paired tiles of 128 rows ----
    p.persist = 0;
    p.psplit = 0;
    const bool geglu = a->epilogue == B200SD_EPI_GEGLU;
    // ---- ... and its split-K mode for the few-tile / deep-K layers the policy above would hand to a split cluster: up to 16
    // K slices per tile, one CTA per slice, partials through an L2-resident workspace (persist_epilogue_split) ----
    if (persist_enabled() && a->split_k <= 0 && a->block_n <= 0 && split > 1 && !geglu && p.rows_valid == BLOCK_M &&
        a->N % 32 == 0 && a->workspace != nullptr && a->workspace_bytes >= kWsPartialBytes + kWsCounterBytes &&
        (reinterpret_cast<uintptr_t>(a->workspace) & 127) == 0 && a->ldc % 4 == 0 && (!a->residual || a->ldr % 4 == 0)) {
        int bnp = 0;
        for (int cand : {160, 128, 256, 192, 96, 64, 32})
            if (a->N % cand == 0) { bnp = cand; break; }
        const int sms_s = b200sd_num_sms();
        const long tiles = bnp ? (long)m_tiles * (a->N / bnp) : sms_s + 1;
        int S = 1;
        while (S < 16 && tiles * (S * 2) <= sms_s && p.num_k_blocks / (S * 2) >= 4) S *= 2;
        // Measured with cold weights (tools/cold_probe.py): the trip through the workspace and the counter costs ~6 us, more
        // than the DSMEM exchange of a split cluster (~4 us) -- it only pays where 16 slices put twice as many SMs on the weight
        // stream as a cluster of 8 can: the 8x8 level (M = 128: 8 tiles; K 23040: 31.2 -> 22.5 us).  Elsewhere (M 512 K 1280:
        // 10.1 -> 15.9 us) the cluster path stays.
        if (S == 16 && p.num_k_blocks >= 128) {
            p.persist = 1;
            p.psplit = S;
            p.block_n = bnp;
            p.split_k = 1;
            p.pair = 0;
            *n_tiles_out = a->N / bnp;
            return B200SD_OK;
        }
    }
    if (persist_enabled() && split == 1 && !p.pair && p.rows_valid == BLOCK_M && a->N % 32 == 0 &&
        (!a->rowbias || (a->rows_per_image > 0 && a->rows_per_image % 32 == 0)) &&
        !(a->residual && a->residual == a->out && a->residual_dtype != a->out_dtype)) {
        const int bnp = a->block_n > 0 ? a->block_n : pick_block_n_persist(a->N, m_tiles, geglu);
        // WHERE the persistent kernel is used.  Measured on B200 inside the real step and with a cold-weight probe
        // (tools/cold_probe.py: every launch reads a different copy of the weights, as in the step where 1.7 GB of weights
        // stream through the 126 MB L2): it wins where a CTA walks >= 2 tiles -- GEGLU feed-forward M8192 N2560 K320 35.0 ->
        // 23.4 us, M2048 N5120 K640 24.4 -> 21.8, fused QKV M8192 N960 K320 14.8 -> 12.2 -- because the epilogue of tile i
        // overlaps the main loop of tile i+1 and no CTA is launched / set up per tile.  On one-tile-per-CTA grids (<= 148
        // tiles) the critical path is load latency -> MMAs -> epilogue either way, the deeper ring of gemm_tcgen05_kernel
        // (5-6 stages: nothing of its smem is set aside for epilogue chunks) hides the HBM latency of the cold weights better,
        // and the persistent kernel measured level or slower (M8192 N320 K1280 12.4 -> 14.1 us): those grids stay there
        // unless debug key 0 forces the persistent kernel.
        const long ptiles = bnp > 0 ? (long)m_tiles * (a->N / bnp) : 0;
        const bool multi = ptiles >= 2L * b200sd_num_sms();
        if (bnp > 0 && bnp <= 256 && bnp % (geglu ? 64 : 32) == 0 && a->N % bnp == 0 && (multi || g_persist > 0)) {
            p.persist = 1;
            p.block_n = bnp;
            *n_tiles_out = a->N / bnp;
        }
    }
    return B200SD_OK;
}

extern "C" int b200sd_gemm(const b200sd_gemm_args* a, b200sd_stream_t stream) {
    B200SD_REQUIRE(a != nullptr, "gemm: null args");
    B200SD_REQUIRE(a->a0 && a->w && a->out, "gemm: null operand pointer");
    B200SD_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, "gemm: non-positive dims M=%d N=%d K=%d", a->M, a->N, a->K);
    B200SD_REQUIRE(a->conv_taps == 1 || a->conv_taps == 9, "gemm: conv_taps must be 1 or 9");
    const int C0 = a->C0, C1 = a->a1 ? a->C1 : 0, C = C0 + C1;
    B200SD_REQUIRE(C0 > 0 && C0 % BLOCK_K == 0 && C1 % BLOCK_K == 0, "gemm: channel counts must be multiples of 64 (C0=%d C1=%d)", C0, C1);
    B200SD_REQUIRE(a->K == a->conv_taps * C, "gemm: K=%d != taps*C=%d", a->K, a->conv_taps * C);
    B200SD_REQUIRE(a->N % 16 == 0, "gemm: N=%d must be a multiple of 16", a->N);
    B200SD_REQUIRE(a->epilogue == B200SD_EPI_LINEAR || a->epilogue == B200SD_EPI_GEGLU, "gemm: bad epilogue");
    B200SD_REQUIRE(a->epilogue != B200SD_EPI_GEGLU || (a->bias && !a->residual && !a->rowbias && a->out_dtype == B200SD_BF16),
                   "gemm: GEGLU epilogue needs bias, bf16 out and no residual/rowbias");
    B200SD_REQUIRE(a->out_dtype == B200SD_BF16 || a->out_dtype == B200SD_F32, "gemm: bad out dtype");
    B200SD_REQUIRE(a->residual_dtype == B200SD_BF16 || a->residual_dtype == B200SD_F32, "gemm: bad residual dtype");
    B200SD_REQUIRE(a->ldc % 8 == 0 && (!a->residual || a->ldr % 8 == 0), "gemm: ldc/ldr must be multiples of 8");
    B200SD_REQUIRE((reinterpret_cast<uintptr_t>(a->out) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->a0) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(a->w) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->a1) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(a->residual) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->bias) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(a->rowbias) & 15) == 0,
                   "gemm: pointers must be 16-byte aligned");
    B200SD_REQUIRE(!a->rowbias || (a->rows_per_image > 0 && a->ldrb % 4 == 0), "gemm: rowbias needs rows_per_image and ldrb %% 4 == 0");

    KParams p;
    memset(&p, 0, sizeof(p));
    p.M = a->M;
    p.N = a->N;
    p.num_k_blocks = a->K / BLOCK_K;
    p.conv = a->conv_taps == 9;
    p.cblocks0 = C0 / BLOCK_K;
    p.cblocks = C / BLOCK_K;
    p.bias = a->bias;
    p.rowbias = a->rowbias;
    p.residual = a->residual;
    p.res_f32 = a->residual_dtype == B200SD_F32;
    p.out = a->out;
    p.ldc = a->ldc;
    p.ldr = a->ldr;
    p.ldrb = a->ldrb > 0 ? a->ldrb : a->N;
    p.rows_per_image = a->rows_per_image > 0 ? a->rows_per_image : 1;
    p.epilogue = a->epilogue;
    p.out_f32 = a->out_dtype == B200SD_F32;
    p.conv_sign = 1;
    p.n_valid = a->N;
    p.tiles_per_tap = 1;

    int m_tiles = 0, n_tiles = 0;
    {
        const int rc = gemm_tiling(a, p, &m_tiles, &n_tiles);
        if (rc) return rc;
    }
    const int bn = p.block_n, split = p.split_k;
    p.gn_part = a->gn_part;
    B200SD_REQUIRE(!a->gn_part || (a->out_dtype == B200SD_F32 && a->epilogue == B200SD_EPI_LINEAR &&
                                   (!a->residual || a->residual_dtype == B200SD_F32)),
                   "gemm: gn_part needs fp32 output, the linear epilogue and no bf16 residual");

    // ---- tensor maps ----
    if (!p.conv) {
        const uint64_t dimsA[2] = {(uint64_t)C0, (uint64_t)a->M};
        const uint64_t strA[2] = {0, (uint64_t)(a->lda0 > 0 ? a->lda0 : C0) * 2};
        const uint32_t boxA[2] = {BLOCK_K, BLOCK_M};
        int rc = b200sd_make_tmap(&p.tmA0, a->a0, 2, dimsA, strA, boxA, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
        if (C1 > 0) {
            const uint64_t dimsA1[2] = {(uint64_t)C1, (uint64_t)a->M};
            const uint64_t strA1[2] = {0, (uint64_t)(a->lda1 > 0 ? a->lda1 : C1) * 2};
            rc = b200sd_make_tmap(&p.tmA1, a->a1, 2, dimsA1, strA1, boxA, CU_TENSOR_MAP_SWIZZLE_128B);
            if (rc) return rc;
        }
    } else {
        const uint32_t boxA[4] = {BLOCK_K, (uint32_t)p.tile_w, (uint32_t)p.tile_h, (uint32_t)p.tile_n};
        const uint64_t dims0[4] = {(uint64_t)C0, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->batch};
        const uint64_t str0[4] = {0, (uint64_t)C0 * 2, (uint64_t)a->W * C0 * 2, (uint64_t)a->H * a->W * C0 * 2};
        int rc = b200sd_make_tmap(&p.tmA0, a->a0, 4, dims0, str0, boxA, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
        if (C1 > 0) {
            const uint64_t dims1[4] = {(uint64_t)C1, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->batch};
            const uint64_t str1[4] = {0, (uint64_t)C1 * 2, (uint64_t)a->W * C1 * 2, (uint64_t)a->H * a->W * C1 * 2};
            rc = b200sd_make_tmap(&p.tmA1, a->a1, 4, dims1, str1, boxA, CU_TENSOR_MAP_SWIZZLE_128B);
            if (rc) return rc;
        }
    }
    {
        const uint64_t dimsB[2] = {(uint64_t)a->K, (uint64_t)a->N};
        const uint64_t strB[2] = {0, (uint64_t)a->K * 2};
        const uint32_t boxB[2] = {BLOCK_K, (uint32_t)(p.pair ? bn / 2 : bn)};
        int rc = b200sd_make_tmap(&p.tmB, a->w, 2, dimsB, strB, boxB, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }

    if (p.persist) return launch_persist(a, p, m_tiles, stream);
    return launch_gemm(p, m_tiles, n_tiles, split, /*cluster=*/true, stream);
}

// Layout of the GroupNorm column statistics a GEMM with these arguments writes into gn_part: partial row
// (m_tile * split_k + rank) holds [sum | sum of squares][N] over the output rows that CTA stored; image b owns the rows
// [b * parts_per_image, (b + 1) * parts_per_image).  parts_per_image == 0: tiles of this shape straddle images (or the
// shape is otherwise not covered) -- do not pass gn_part.  hw = output rows per image.
extern "C" int b200sd_gemm_gn_layout(const b200sd_gemm_args* a, int hw, int* parts_per_image, int* total_parts) {
    B200SD_REQUIRE(a && parts_per_image && total_parts && hw > 0, "gemm_gn_layout: bad arguments");
    KParams p;
    memset(&p, 0, sizeof(p));
    p.M = a->M;
    p.N = a->N;
    p.num_k_blocks = a->K / BLOCK_K;
    p.conv = a->conv_taps == 9;
    int m_tiles = 0, n_tiles = 0;
    const int rc = gemm_tiling(a, p, &m_tiles, &n_tiles);
    if (rc) return rc;
    *parts_per_image = 0;
    *total_parts = 0;
    if (a->out_dtype != B200SD_F32 || a->epilogue != B200SD_EPI_LINEAR || (a->residual && a->residual_dtype != B200SD_F32)) return B200SD_OK;
    if (p.persist && p.psplit > 1) {
        // split-K mode: one partial row per (tile, K slice) = 128 / split output rows
        const int rpc = BLOCK_M / p.psplit;
        if (a->M % hw != 0 || hw % rpc != 0 || (p.conv && a->H * a->W != hw)) return B200SD_OK;
        *parts_per_image = hw / rpc;
        *total_parts = m_tiles * p.psplit;
        return B200SD_OK;
    }
    if (p.persist) {
        // the persistent kernel publishes one partial row per 128-row tile
        if (a->M % hw != 0 || hw % BLOCK_M != 0 || (p.conv && a->H * a->W != hw)) return B200SD_OK;
        *parts_per_image = hw / BLOCK_M;
        *total_parts = m_tiles;
        return B200SD_OK;
    }
    // Partial row (m_tile * split + rank) covers the BLOCK_M / split output rows that rank stores; it is usable when those
    // rows never straddle two images and the partial rows of an image are contiguous.
    const int rpp = BLOCK_M / p.split_k;     // rows per partial
    int ppi;
    if (p.conv) {
        if (a->H * a->W != hw) return B200SD_OK;
        if (p.tile_n == 1) ppi = p.tiles_y * p.tiles_x * p.split_k;              // tiles inside one image (empty ranks publish zeros)
        else if (p.rows_valid == BLOCK_M && hw % rpp == 0) ppi = hw / rpp;   // whole images per tile, split finer than an image
        else return B200SD_OK;
    } else {
        if (a->M % hw != 0 || hw % rpp != 0) return B200SD_OK;
        ppi = hw / rpp;
    }
    if (p.pair) m_tiles = (m_tiles + 1) & ~1;
    *parts_per_image = ppi;
    *total_parts = m_tiles * p.split_k;
    return B200SD_OK;
}

// ------------------------------------------------------------------------------------------------
// backward entry points (same kernel, MN-major operand modes)
// ------------------------------------------------------------------------------------------------
extern "C" int b200sd_gemm_dgrad(const b200sd_dgrad_args* a, b200sd_stream_t stream) {
    B200SD_REQUIRE(a != nullptr && a->dy && a->w && a->out, "dgrad: null pointer");
    B200SD_REQUIRE(a->conv_taps == 1 || a->conv_taps == 9, "dgrad: conv_taps must be 1 or 9");
    B200SD_REQUIRE(a->M > 0 && a->Cout > 0 && a->Cout % BLOCK_K == 0, "dgrad: Cout=%d must be a positive multiple of 64", a->Cout);
    B200SD_REQUIRE(a->Cin > 0 && a->Cin % 8 == 0, "dgrad: Cin=%d must be a multiple of 8", a->Cin);
    B200SD_REQUIRE(a->out_dtype == B200SD_BF16 || a->out_dtype == B200SD_F32, "dgrad: bad out dtype");
    const int ldy = a->ldy > 0 ? a->ldy : a->Cout;
    const int ldc = a->ldc > 0 ? a->ldc : a->Cin;
    const int ldr = a->ldr > 0 ? a->ldr : a->Cin;
    B200SD_REQUIRE(ldc % 8 == 0 && ldr % 8 == 0 && ldy % 8 == 0, "dgrad: pitches must be multiples of 8");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(a->dy) | reinterpret_cast<uintptr_t>(a->w) | reinterpret_cast<uintptr_t>(a->out) |
                     reinterpret_cast<uintptr_t>(a->residual)) & 15) == 0, "dgrad: pointers must be 16-byte aligned");
    KParams p;
    memset(&p, 0, sizeof(p));
    p.M = a->M;
    p.N = a->Cin;
    p.n_valid = a->Cin;
    p.tiles_per_tap = 1;
    p.conv = a->conv_taps == 9;
    p.conv_sign = -1;
    p.b_mode = 1;
    p.cblocks0 = p.cblocks = a->Cout / BLOCK_K;
    p.num_k_blocks = a->conv_taps * p.cblocks;
    p.residual = a->residual;
    p.res_f32 = a->residual_dtype == B200SD_F32;
    p.out = a->out;
    p.ldc = ldc;
    p.ldr = ldr;
    p.ldrb = a->Cin;
    p.rows_per_image = 1;
    p.epilogue = B200SD_EPI_LINEAR;
    p.out_f32 = a->out_dtype == B200SD_F32;
    int m_tiles;
    if (!p.conv) {
        p.rows_valid = BLOCK_M;
        p.a_bytes = kABytes;
        p.tile_w = p.tile_h = p.tile_n = p.tiles_y = 1;
        p.tiles_x = 1;
        m_tiles = ceil_div(a->M, BLOCK_M);
    } else {
        B200SD_REQUIRE(ldy == a->Cout, "dgrad(conv): dy must be dense NHWC");
        const int rc = conv_m_tiling(p, a->batch, a->H, a->W, a->M, &m_tiles);
        if (rc) return rc;
    }
    int bn = a->block_n > 0 ? a->block_n : pick_block_n_mn(a->Cin, m_tiles, 0);
    B200SD_REQUIRE(bn % 64 == 0 && bn >= 64 && bn <= 256, "dgrad: block_n %d must be 64, 128, 192 or 256", bn);
    p.pair = want_pair(a->pair, 1, m_tiles, ceil_div(a->Cin, bn), p.num_k_blocks);
    if (p.pair && bn % 128 != 0) {
        // a pair splits the 64-column boxes of the B tile evenly: 128 or 256 wide, whichever pads N less
        if (a->block_n > 0) p.pair = 0;
        else bn = (ceil_div(a->Cin, 256) * 256 <= ceil_div(a->Cin, 128) * 128) ? 256 : 128;
    }
    p.block_n = bn;
    const int n_tiles = ceil_div(a->Cin, bn);
    p.tmem_cols = pow2_cols(bn);
    // split-K clusters for the few-tile / deep-K layers (the 8x8 and 16x16 levels), same policy as the forward GEMM
    int split = 1;
    {
        const int sms = b200sd_num_sms();
        const int tiles = m_tiles * n_tiles;
        if (!p.pair && tiles * 2 <= sms && p.num_k_blocks >= 16) {
            while (split < 8 && tiles * split * 2 <= sms && p.num_k_blocks / (split * 2) >= 8) split *= 2;
            if (split == 8 && tiles > 8) split = 4;
        }
    }
    p.split_k = split;
    p.kb_per_split = ceil_div(p.num_k_blocks, split);
    while (split > 1 && (split - 1) * p.kb_per_split >= p.num_k_blocks) {   // never an empty split
        split /= 2;
        p.split_k = split;
        p.kb_per_split = ceil_div(p.num_k_blocks, split);
    }
    int rc;
    if (!p.conv) {
        const uint64_t dimsA[2] = {(uint64_t)a->Cout, (uint64_t)a->M};
        const uint64_t strA[2] = {0, (uint64_t)ldy * 2};
        const uint32_t boxA[2] = {BLOCK_K, BLOCK_M};
        if ((rc = b200sd_make_tmap(&p.tmA0, a->dy, 2, dimsA, strA, boxA, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
        const uint64_t dimsB[2] = {(uint64_t)a->Cin, (uint64_t)a->Cout};
        const uint64_t strB[2] = {0, (uint64_t)a->Cin * 2};
        const uint32_t boxB[2] = {64, BLOCK_K};
        if ((rc = b200sd_make_tmap(&p.tmB, a->w, 2, dimsB, strB, boxB, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    } else {
        const uint32_t boxA[4] = {BLOCK_K, (uint32_t)p.tile_w, (uint32_t)p.tile_h, (uint32_t)p.tile_n};
        const uint64_t dims0[4] = {(uint64_t)a->Cout, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->batch};
        const uint64_t str0[4] = {0, (uint64_t)a->Cout * 2, (uint64_t)a->W * a->Cout * 2, (uint64_t)a->H * a->W * a->Cout * 2};
        if ((rc = b200sd_make_tmap(&p.tmA0, a->dy, 4, dims0, str0, boxA, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
        const uint64_t dimsB[3] = {(uint64_t)a->Cin, 9, (uint64_t)a->Cout};
        const uint64_t strB[3] = {0, (uint64_t)a->Cin * 2, (uint64_t)9 * a->Cin * 2};
        const uint32_t boxB[3] = {64, 1, BLOCK_K};
        if ((rc = b200sd_make_tmap(&p.tmB, a->w, 3, dimsB, strB, boxB, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    }
    return launch_gemm(p, m_tiles, n_tiles, p.split_k, /*cluster=*/true, stream);
}

extern "C" int b200sd_gemm_wgrad(const b200sd_wgrad_args* a, b200sd_stream_t stream) {
    B200SD_REQUIRE(a != nullptr && a->dy && a->x && a->dw, "wgrad: null pointer");
    B200SD_REQUIRE(a->conv_taps == 1 || a->conv_taps == 9, "wgrad: conv_taps must be 1 or 9");
    B200SD_REQUIRE(a->rows > 0 && a->Cout > 0 && a->Cin > 0 && a->Cout % 8 == 0 && a->Cin % 8 == 0,
                   "wgrad: rows=%d Cout=%d Cin=%d (channel counts must be multiples of 8)", a->rows, a->Cout, a->Cin);
    const int ldy = a->ldy > 0 ? a->ldy : a->Cout;
    const int ldx = a->ldx > 0 ? a->ldx : a->Cin;
    const int lddw = a->lddw > 0 ? a->lddw : a->conv_taps * a->Cin;
    B200SD_REQUIRE(ldy % 8 == 0 && ldx % 8 == 0 && lddw % 4 == 0, "wgrad: pitches must be multiples of 8 (dw: 4)");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(a->dy) | reinterpret_cast<uintptr_t>(a->x) | reinterpret_cast<uintptr_t>(a->dw)) & 15) == 0,
                   "wgrad: pointers must be 16-byte aligned");
    KParams p;
    memset(&p, 0, sizeof(p));
    p.M = a->Cout;
    p.N = a->conv_taps * a->Cin;
    p.n_valid = a->Cin;
    p.a_mn = 1;
    p.b_mode = a->conv_taps == 9 ? 3 : 2;
    p.conv = 0;
    p.conv_sign = 1;
    p.rows_valid = BLOCK_M;
    p.a_bytes = kABytes;
    p.out = a->dw;
    p.ldc = lddw;
    p.ldrb = p.N;
    p.rows_per_image = 1;
    p.epilogue = B200SD_EPI_LINEAR;
    p.out_f32 = 1;
    p.atomic_out = 1;
    p.split_k = 1;
    const int m_tiles = ceil_div(a->Cout, BLOCK_M);
    int rc;
    if (a->conv_taps == 9) {
        const int H = a->H, W = a->W, NB = a->batch;
        B200SD_REQUIRE(NB > 0 && H > 0 && W > 0 && a->rows == NB * H * W, "wgrad(conv): rows=%d != batch*H*W", a->rows);
        B200SD_REQUIRE(W <= 64 && 64 % W == 0, "wgrad(conv): W=%d must divide 64", W);
        B200SD_REQUIRE(ldy == a->Cout && ldx == a->Cin, "wgrad(conv): dy / x must be dense NHWC");
        p.tiles_x = 1;
        p.tile_w = W;
        p.tile_h = (64 / W < H) ? 64 / W : H;
        B200SD_REQUIRE(H % p.tile_h == 0, "wgrad(conv): H=%d not a multiple of the %d-row pixel block", H, p.tile_h);
        p.tile_n = 64 / (W * p.tile_h);
        p.tiles_y = H / p.tile_h;
        p.num_k_blocks = p.tile_n > 1 ? ceil_div(NB, p.tile_n) : NB * p.tiles_y;
        const uint32_t boxB[4] = {64, (uint32_t)p.tile_w, (uint32_t)p.tile_h, (uint32_t)p.tile_n};
        const uint64_t dims[4] = {(uint64_t)a->Cin, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
        const uint64_t str[4] = {0, (uint64_t)a->Cin * 2, (uint64_t)W * a->Cin * 2, (uint64_t)H * W * a->Cin * 2};
        if ((rc = b200sd_make_tmap(&p.tmB, a->x, 4, dims, str, boxB, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    } else {
        p.tile_w = p.tile_h = p.tile_n = p.tiles_y = 1;
        p.tiles_x = 1;
        p.num_k_blocks = ceil_div(a->rows, BLOCK_K);
        const uint64_t dimsB[2] = {(uint64_t)a->Cin, (uint64_t)a->rows};
        const uint64_t strB[2] = {0, (uint64_t)ldx * 2};
        const uint32_t boxB[2] = {64, BLOCK_K};
        if ((rc = b200sd_make_tmap(&p.tmB, a->x, 2, dimsB, strB, boxB, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    }
    {
        const uint64_t dimsA[2] = {(uint64_t)a->Cout, (uint64_t)a->rows};
        const uint64_t strA[2] = {0, (uint64_t)ldy * 2};
        const uint32_t boxA[2] = {64, BLOCK_K};
        if ((rc = b200sd_make_tmap(&p.tmA0, a->dy, 2, dimsA, strA, boxA, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    }
    const int bn = a->block_n > 0 ? a->block_n : pick_block_n_mn(a->Cin, m_tiles * a->conv_taps, a->conv_taps == 9 ? 2 : 1);
    B200SD_REQUIRE(bn % 64 == 0 && bn >= 64 && bn <= 256, "wgrad: block_n %d must be 64, 128, 192 or 256", bn);
    p.block_n = bn;
    p.tiles_per_tap = ceil_div(a->Cin, bn);
    const int n_tiles = a->conv_taps * p.tiles_per_tap;
    p.tmem_cols = pow2_cols(bn);
    // split-K over grid.z (fp32 red.add combines the partials): aim at >= 2 CTAs per SM, >= 8 k-blocks per split
    int split = a->split_k;
    if (split <= 0) {
        const int tiles = m_tiles * n_tiles;
        split = ceil_div(2 * b200sd_num_sms(), tiles);
        const int max_split = p.num_k_blocks / 8 > 0 ? p.num_k_blocks / 8 : 1;
        if (split > max_split) split = max_split;
        if (split < 1) split = 1;
    }
    if (split > p.num_k_blocks) split = p.num_k_blocks;
    p.kb_per_split = ceil_div(p.num_k_blocks, split);
    split = ceil_div(p.num_k_blocks, p.kb_per_split);   // no empty splits
    return launch_gemm(p, m_tiles, n_tiles, split, false, stream);
}
