/* b200sd.h -- C ABI of libb200sd.so: the sm_100a (B200) kernels behind the SD v1.x UNet denoise
 * hot path (UNet2DConditionModel.forward, scheduler.step / add_noise, CFG combine, MSE loss).
 *
 * The reference (Edenzzzz/Stable-Diffusion-for-book-cover-generation) has no FFI of its own: the
 * boundary is the diffusers 0.7.2 Python class surface.  Every entry point below names the
 * reference call site whose arithmetic it replaces; the Python facade in
 * `stable-diffusion-for-book-cover-generation_b200/` (import name `b200sd`) binds them with ctypes
 * (INTEGRATION.md shows the binding a maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise;
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*), never synchronises,
 *     never allocates: scratch is caller-provided (`*_workspace_bytes` says how much);
 *   - return 0 on success, non-zero (B200SD_ERR_*) on error; b200sd_last_error() gives the text;
 *   - activations are NHWC ("channels last"): a (N,C,H,W) tensor is stored as [N*H*W][C];
 *   - dtype codes: B200SD_F32 = 0, B200SD_BF16 = 1.
 */
#ifndef B200SD_H_
#define B200SD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SD_OK 0
#define B200SD_ERR_INVALID 1
#define B200SD_ERR_CUDA 2
#define B200SD_ERR_UNSUPPORTED 3

#define B200SD_F32 0
#define B200SD_BF16 1

typedef void* b200sd_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------------------------- */
const char* b200sd_last_error(void);
int b200sd_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t b200sd_launch_count(void);

/* In-graph timers (measurement plumbing, SURVEY.md 8d): process-wide CUDA events.  b200sd_timer_record(i) records event i on
 * `stream`; while the stream is being captured the record becomes an external event-record node, so a replay of the captured
 * plan timestamps the gaps between its kernels and b200sd_timer_elapsed_ms(i, j) gives per-kernel times inside the real step. */
/* debug override of the GEMM launch policy: key 0 = persistent kernel (-1 default, 0 off, 1 on); other keys are ignored */
void b200sd_debug_set(int key, int value);
int b200sd_timer_reserve(int n);
int b200sd_timer_record(int i, b200sd_stream_t stream);
int b200sd_timer_elapsed_ms(int i, int j, float* ms);

/* ---- scheduler / loss elementwise kernels (HBM-bound) ------------------------------------- */

/* Classifier-free-guidance combine fused with the DDIM update (eta = 0):
 *   eps = eps_u + g (eps_c - eps_u);  x0 = (x - sb_t eps) / sa_t;  out = sa_p x0 + sb_p eps
 * Replaces the pipeline's `noise_pred_uncond + guidance_scale * (...)` and DDIMScheduler.step
 * (reference call sites inference.py:175-176, 386-387; SURVEY.md App. B.2/B.4).
 * eps_c == NULL -> no CFG (eps = eps_u).  eps_out must be NULL: since version 102 the combined eps is not written out and a
 * non-NULL eps_out returns B200SD_ERR_INVALID.  This is b200sd_cfg_ancestral_step with c_x0 = sa_p, c_x = 0, c_e = sb_p, no
 * noise and no clipping, whose error messages it returns.
 * x_dtype / eps_dtype: B200SD_F32 or B200SD_BF16; out has x_dtype.  out may alias x.
 * Algorithmic bytes: 4 * n * elem (3 reads + 1 write). */
int b200sd_cfg_ddim_step(const void* eps_u, const void* eps_c, const void* x, void* out, void* eps_out,
                         int64_t n, float guidance, float sa_t, float sb_t, float sa_p, float sb_p,
                         int eps_dtype, int x_dtype, b200sd_stream_t stream);

/* Captured sampler: the whole denoising step (timestep -> UNet plan -> CFG + scheduler update) is ONE CUDA graph that is
 * replayed with no host-side arguments, so the step index lives on the device.  `cursor` is int[2]: [0] = next step, [1] = the
 * step being executed.  b200sd_sampler_advance opens a step: in_t[0..n_t) = timesteps[cursor[0]] (the UNet plan's timestep
 * input), cursor[1] = cursor[0], cursor[0] = (cursor[0] + 1) % n_steps.  b200sd_cfg_ancestral_step_table (DDIM, DDPM) or
 * b200sd_cfg_plms_step_table (PLMS) closes it with the coefficients of row cursor[1] of its table.  Replaces the per-step
 * Python of StableDiffusionPipeline.__call__'s loop (reference call sites inference.py:175-176, 342-351). */
int b200sd_sampler_advance(const float* timesteps, int n_steps, int* cursor, float* in_t, int n_t, b200sd_stream_t stream);

/* The PLMS step of the captured sampler (fp32): x (the latents) is updated in place; `saved` (n floats) holds the
 * sample of the first call for PNDM's repeated first timestep; `ring` is the 4-deep eps history (4 * n floats).  Per call one
 * row of 12 floats of `table`, indexed by cursor[1]: w0 w1 w2 w3 | cx ce | h1 h2 h3 (ring slot of ets[-1], ets[-2], ets[-3];
 * -1 = unused) | out_slot (-1 = this call's eps is not kept) | x_from_saved | save_x.  The host fills the table by running
 * PNDMScheduler's counter logic once (sampler.py); reference call site utils.py:222-224. */
int b200sd_cfg_plms_step_table(const float* eps_u, const float* eps_c, float* x, float* saved, float* ring, int64_t n,
                               float guidance, const float* table, const int* cursor, b200sd_stream_t stream);

/* CFG combine fused with the affine update of DDPMScheduler.step and DDIMScheduler.step (any eta in [0, 1]):
 *   eps = eps_u + g (eps_c - eps_u);  x0 = (x - sb_t eps) / sa_t;  if clip: x0 = clamp(x0, -1, 1)
 *   out = c_x0 x0 + c_x x + c_e eps + (noise ? c_z noise : 0)
 * noise: fp32, n elements, NULL = no noise term (DDIM with eta = 0, DDPM's t = 0 step).  The host draws it from the caller's
 * generator.
 * x_dtype / eps_dtype: B200SD_F32 or B200SD_BF16; out has x_dtype.  out may alias x.
 * Algorithmic bytes: 5 * n * 4 in fp32 (eps_u, eps_c, x, noise read; out written). */
int b200sd_cfg_ancestral_step(const void* eps_u, const void* eps_c, const void* x, const float* noise, void* out,
                              int64_t n, float guidance, float sa_t, float sb_t, float c_x0, float c_x, float c_e, float c_z,
                              int clip, int eps_dtype, int x_dtype, b200sd_stream_t stream);

/* The captured-sampler form of b200sd_cfg_ancestral_step (fp32; x is updated in place), for DDIM and DDPM.  Per step one row
 * of 8 floats of `table` (16-byte aligned), indexed by cursor[1]: sa_t sb_t c_x0 c_x c_e c_z noise_row clip.  noise_row = -1:
 * this step adds no noise and `noise` is not read; otherwise z = noise + noise_row * n (`noise` is [n_noisy_steps][n] floats,
 * filled by the host before the run).  `noise` may be NULL when no row names a noise row. */
int b200sd_cfg_ancestral_step_table(const float* eps_u, const float* eps_c, float* x, const float* noise, int64_t n,
                                    float guidance, const float* table, const int* cursor, b200sd_stream_t stream);

/* CFG combine fused with the PLMS (PNDM skip_prk_steps=True) linear-multistep update:
 *   eps = eps_u + g (eps_c - eps_u);  e = w[0] eps + sum_{i<nhist} w[1+i] hist[i];
 *   out = cx * x - ce * e
 * Replaces PNDMScheduler.step_plms/_get_prev_sample (reference call site utils.py:222-224;
 * SURVEY.md App. B.3).  eps_out (optional) receives eps so the host can keep the 4-deep history.
 * hist pointers are device pointers with eps_dtype elements. */
int b200sd_cfg_plms_step(const void* eps_u, const void* eps_c, const void* x, void* out, void* eps_out,
                         const void* hist0, const void* hist1, const void* hist2, const void* hist3,
                         int nhist, const float* w_host5, int64_t n, float guidance, float cx, float ce,
                         int eps_dtype, int x_dtype, b200sd_stream_t stream);

/* DDPMScheduler.add_noise (finetune_sd.py:473-474): out[b] = sa[t[b]] x0[b] + sb[t[b]] noise[b].
 * timesteps: int64[batch] (device); sa_table / sb_table: float[num_train_timesteps] (device). */
int b200sd_add_noise(const void* x0, const void* noise, const int64_t* timesteps, const float* sa_table,
                     const float* sb_table, void* out, int batch, int64_t per_sample, int num_train_timesteps,
                     int dtype, b200sd_stream_t stream);

/* The masking step of legacy inpainting (diffusers 0.7.2 StableDiffusionInpaintPipelineLegacy), run after every scheduler step
 * at loop timestep t, fp32 and in place:
 *   x = m (sa[t] x0 + sb[t] noise) + (1 - m) x
 * x, x0 (the init latents before noising), noise (the init noise) and m (1 = keep, not binarised) all have n elements: the
 * host expands the mask to the latents' shape.  sa_table / sb_table: float[num_train_timesteps], the tables of
 * b200sd_add_noise; t is clamped to [0, num_train_timesteps).  Algorithmic bytes: 5 * n * 4 (x, x0, noise, m read; x written).
 * b200sd_inpaint_blend takes t by value; b200sd_inpaint_blend_table (the captured sampler) reads t = t_table[cursor[1]] on the
 * device, the timestep table and cursor of b200sd_sampler_advance. */
int b200sd_inpaint_blend(float* x, const float* x0, const float* noise, const float* mask, int64_t n, int64_t timestep,
                         const float* sa_table, const float* sb_table, int num_train_timesteps, b200sd_stream_t stream);
int b200sd_inpaint_blend_table(float* x, const float* x0, const float* noise, const float* mask, int64_t n,
                               const float* t_table, const int* cursor, const float* sa_table, const float* sb_table,
                               int num_train_timesteps, b200sd_stream_t stream);

/* F.mse_loss(pred, target, "none").mean([1,2,3]).mean() (finetune_sd.py:483-484) == global mean.
 * loss_out: float[1]; workspace: float[b200sd_mse_workspace_floats()]. */
int b200sd_mse_workspace_floats(void);
int b200sd_mse_loss_fwd(const void* pred, const void* target, float* loss_out, float* workspace, int64_t n,
                        int pred_dtype, int target_dtype, b200sd_stream_t stream);
/* grad_pred = grad_loss[0] * 2 (pred - target) / n ; grad_loss: device float[1] */
int b200sd_mse_loss_bwd(const void* pred, const void* target, const float* grad_loss, void* grad_pred, int64_t n,
                        int pred_dtype, int target_dtype, b200sd_stream_t stream);

/* ---- UNet building blocks ----------------------------------------------------------------- */

/* diffusers Timesteps (flip_sin_to_cos=True, freq_shift=0) (SURVEY.md App. A.2):
 * out[b, 0:dim/2] = cos(t_b f_i), out[b, dim/2:] = sin(t_b f_i), f_i = exp(-ln(1e4) i / (dim/2)).
 * timesteps: float[batch] (device). out: float[batch, dim]. */
int b200sd_timestep_embedding(const float* timesteps, float* out, int batch, int dim, b200sd_stream_t stream);

/* Small-M linear for the time-embedding MLP and the 22 time_emb_proj heads:
 *   out[b, n] = bias[n] + sum_k act(in[b, k]) * W[n, k],  act = SiLU if silu_in else identity,
 *   optional SiLU on the output.  in/out fp32, W bf16 [N,K] row-major, bias fp32. */
int b200sd_small_linear(const float* in, const void* w_bf16, const float* bias, float* out, int batch, int N, int K,
                        int silu_in, int silu_out, b200sd_stream_t stream);

/* GEMM / implicit-GEMM conv on tcgen05 tensor cores (TMA -> smem -> tcgen05.mma -> TMEM).
 *   out[M, N] = A[M, K] * W[N, K]^T  (+ bias[N]) (+ rowbias[row / rows_per_image, N]) (+ residual[M, N])
 * A and W are bf16, accumulation fp32, out bf16 (or fp32 when out_dtype == B200SD_F32).
 * Replaces nn.Linear / Conv2d 1x1 / Conv2d 3x3 (cuBLAS / cuDNN in the reference stack;
 * SURVEY.md section 2.3 K1, K2, K3, K5).
 *
 * A operand:
 *   conv_taps == 1 : plain GEMM. A is [M, C0] (lda0 elements between rows); if a1 != NULL the K
 *                    dimension is the channel concat [a0 | a1] (C0 + C1), i.e. torch.cat fused.
 *   conv_taps == 9 : 3x3 stride-1 pad-1 conv over NHWC [batch, H, W, C0(+C1)];
 *                    K = 9 * (C0 + C1), W is [N][ky][kx][C0+C1]; M = batch * H * W.
 * epilogue:
 *   B200SD_EPI_LINEAR : bias / rowbias / residual as above.
 *   B200SD_EPI_GEGLU  : W rows are tile-interleaved [value | gate] (see b200sd_geglu_tile());
 *                       out[M, N/2] = value * gelu_erf(gate), bias likewise interleaved.
 * split_k in {1, 2, 4, 8}: the split CTAs of a tile form a thread-block cluster, exchange their fp32
 * partial tiles through distributed shared memory and each reduces + stores 128/split_k rows in a fixed
 * order (bit-deterministic).  No scratch is needed (workspace may be NULL).
 */
#define B200SD_EPI_LINEAR 0
#define B200SD_EPI_GEGLU 1

typedef struct b200sd_gemm_args {
    const void* a0;        /* bf16 */
    const void* a1;        /* bf16 or NULL */
    const void* w;         /* bf16 [N, K] */
    const float* bias;     /* [N] or NULL */
    const float* rowbias;  /* [batch, N] or NULL (time-embedding add) */
    const void* residual;  /* [M, ldr] (residual_dtype) or NULL */
    void* out;             /* [M, ldc] */
    int M, N, K;
    int C0, C1;            /* channels of a0 / a1 */
    int lda0, lda1;        /* row pitch (elements) of a0 / a1 in plain-GEMM mode */
    int ldc, ldr;
    int ldrb;              /* row pitch of rowbias (0 = N) */
    int conv_taps;         /* 1 or 9 */
    int batch, H, W;       /* conv geometry (conv_taps == 9) */
    int rows_per_image;    /* for rowbias: image index = row / rows_per_image */
    int epilogue;          /* B200SD_EPI_* */
    int out_dtype;         /* B200SD_BF16 or B200SD_F32 */
    int residual_dtype;    /* B200SD_BF16 or B200SD_F32 */
    int block_n;           /* 0 = auto */
    int split_k;           /* 0 = auto */
    void* workspace;       /* split-K scratch (may be NULL when split_k == 1) */
    size_t workspace_bytes;
    int pair;              /* CTA pairs (tcgen05 cta_group::2, 256-row MMA tiles): 0 = auto, 1 = on, -1 = off */
    float* gn_part;        /* optional: per-CTA column statistics [parts][2][N] of the fp32 output (sum | sum of squares over the
                              rows each CTA stores), consumed by b200sd_groupnorm_silu_parts; layout from b200sd_gemm_gn_layout */
} b200sd_gemm_args;

size_t b200sd_gemm_workspace_bytes(void);
int b200sd_geglu_tile(int N); /* tile width used to interleave GEGLU weights for a given N (= 8C) */
int b200sd_gemm(const b200sd_gemm_args* args, b200sd_stream_t stream);
/* How a GEMM with these arguments lays out gn_part: image b (hw output rows each) owns the partial rows
 * [b * parts_per_image, (b + 1) * parts_per_image) of total_parts.  parts_per_image == 0: not available for this shape
 * (output tiles straddle images, bf16 output, ...) -- leave gn_part NULL and use b200sd_groupnorm_silu. */
int b200sd_gemm_gn_layout(const b200sd_gemm_args* args, int hw, int* parts_per_image, int* total_parts);

/* ---- backward GEMMs (autograd.backward through the UNet, finetune_sd.py:494; SURVEY.md row A9) ----
 * Same tcgen05 pipeline as b200sd_gemm; the operands that the forward read K-major are read MN-major
 * here (UMMA "transpose" descriptors over 64-column SWIZZLE_128B TMA boxes), so neither a transposed
 * weight copy nor a transposed activation copy exists.
 *
 * Data gradient of out = X W^T (conv_taps == 1) or of the 3x3 pad-1 conv (conv_taps == 9):
 *   dX[M, Cin] = sum_tap dY[p - d(tap), :] * W[:, tap, :]   (+ residual)
 * dy: bf16 [M, ldy] (dense NHWC for conv); w: the FORWARD weight, bf16 [Cout][taps][Cin];
 * out: [M, ldc] bf16 / fp32; residual (optional, [M, ldr]) is added -- pass residual == out to accumulate.
 * Cout must be a multiple of 64, Cin a multiple of 8.  Replaces cuBLAS / cuDNN dgrad. */
typedef struct b200sd_dgrad_args {
    const void* dy;
    const void* w;
    const void* residual;
    void* out;
    int M, Cout, Cin;
    int conv_taps;        /* 1 or 9 */
    int batch, H, W;      /* conv geometry */
    int ldy, ldc, ldr;    /* 0 = dense */
    int out_dtype, residual_dtype;
    int block_n;          /* 0 = auto (64 / 128 / 192 / 256) */
    int pair;             /* CTA pairs: 0 = auto, 1 = on, -1 = off */
} b200sd_dgrad_args;
int b200sd_gemm_dgrad(const b200sd_dgrad_args* args, b200sd_stream_t stream);

/* Weight gradient, ACCUMULATED into fp32 (red.global.add: split-K partials and gradient accumulation
 * share the mechanism, so dw must hold the running gradient -- zero it at the start of a step):
 *   dW[Cout][tap][Cin] += sum_p dY[p, co] * X[p + d(tap), ci]
 * dy: bf16 [rows, ldy]; x: bf16 [rows, ldx] (dense NHWC [batch,H,W,Cin] for conv, W | 64);
 * dw: fp32 [Cout][lddw] (lddw = taps * Cin when 0).  Replaces cuBLAS / cuDNN wgrad. */
typedef struct b200sd_wgrad_args {
    const void* dy;
    const void* x;
    float* dw;
    int rows, Cout, Cin;
    int conv_taps;
    int batch, H, W;
    int ldy, ldx, lddw;
    int block_n, split_k; /* 0 = auto */
} b200sd_wgrad_args;
int b200sd_gemm_wgrad(const b200sd_wgrad_args* args, b200sd_stream_t stream);

/* Direct 3x3 convs at the ends of the UNet (degenerate GEMM shapes, CUDA cores):
 * conv_in : NCHW fp32 (batch, Cin=4, H, W) -> NHWC bf16 (batch*H*W, Cout); w fp32 packed [Cout][ky][kx][Cin].
 * conv_out: NHWC bf16 (batch*H*W, Cin) -> NCHW fp32 (batch, Cout<=4, H, W); w fp32 packed [Cout][ky][kx][Cin]. */
int b200sd_conv_in(const float* x_nchw, const float* w, const float* bias, void* out_nhwc, int batch, int Cin,
                   int Cout, int H, int W, int out_dtype, b200sd_stream_t stream);
int b200sd_conv_out(const void* x_nhwc, const float* w, const float* bias, float* out_nchw, int batch, int Cin,
                    int Cout, int H, int W, b200sd_stream_t stream);
/* Tail of conv_out when it runs as an implicit GEMM on the tensor cores (large batches: b200sd_gemm with the 4 output channels
 * padded to a 32-wide tile and the fp32 weights split into bf16 hi | lo halves along K): x fp32 [batch*hw][ld] NHWC, the first C
 * (<= 4) columns are the channels; out_nchw[b][c][p] = x[b*hw + p][c] + bias[c]. */
int b200sd_nhwc_bias_to_nchw(const float* x, const float* bias, float* out_nchw, int batch, int C, int hw, int ld,
                             b200sd_stream_t stream);

/* GroupNorm over NHWC input, optionally over the channel concat [x0 | x1] (torch.cat fused),
 * optional SiLU, bf16 output [rows, C0+C1].  stats_ws: float[b200sd_groupnorm_workspace_floats(batch)]
 * scratch that must be ZERO before its first use (arrival counters; the kernels leave them zeroed).
 * x0 / x1 have in_dtype (fp32 residual stream or bf16); raw_out (optional, bf16 [rows, C0+C1]) receives the
 * un-normalised concat, the operand of the 1x1 shortcut conv.
 * Replaces nn.GroupNorm + SiLU (+ torch.cat) in ResnetBlock2D / Transformer2DModel. */
int b200sd_groupnorm_silu(const void* x0, const void* x1, int C0, int C1, const float* gamma, const float* beta,
                          void* out, void* raw_out, float* stats_ws, int batch, int hw, int groups, float eps,
                          int silu, int in_dtype, b200sd_stream_t stream);

/* Same, additionally writing stats_out[batch][groups][2] = (mean, rstd) per (image, group) for the backward pass
 * (stats_out may be NULL). */
int b200sd_groupnorm_silu_stats(const void* x0, const void* x1, int C0, int C1, const float* gamma, const float* beta,
                                void* out, void* raw_out, float* stats_ws, float* stats_out, int batch, int hw, int groups,
                                float eps, int silu, int in_dtype, b200sd_stream_t stream);

/* GroupNorm (+SiLU, + concat) whose statistics come from the GEMMs that PRODUCED x0 / x1 (b200sd_gemm_args::gn_part,
 * layout from b200sd_gemm_gn_layout: part [image][ppi][2][ld] floats): no statistics pass over the tensor.  Same
 * semantics as b200sd_groupnorm_silu_stats otherwise.  Returns B200SD_ERR_UNSUPPORTED for channel layouts it does not
 * cover -- fall back to b200sd_groupnorm_silu. */
int b200sd_groupnorm_silu_parts(const void* x0, const void* x1, int C0, int C1, const float* part0, int ppi0, int ld0,
                                const float* part1, int ppi1, int ld1, const float* gamma, const float* beta, void* out,
                                void* raw_out, float* stats_out, int batch, int hw, int groups, float eps, int silu,
                                int in_dtype, b200sd_stream_t stream);

/* LayerNorm over the last dim of [rows, C] (in_dtype: fp32 or bf16) -> bf16 (affine). */
int b200sd_groupnorm_workspace_floats(int batch);
int b200sd_layernorm(const void* x, const float* gamma, const float* beta, void* out, int rows, int C, float eps,
                     int in_dtype, b200sd_stream_t stream);

/* Fused (flash-style) attention: out = softmax(scale * Q K^T) V per (batch, head).
 * q: [batch*Sq, ldq] with head h at columns [h*d, (h+1)*d); k, v likewise with ldk / ldv;
 * out: [batch*Sq, ldo].  All bf16, fp32 softmax/accumulate.  d in {40, 80, 160} (+ 32, 64, 128).
 * Head dims 40 / 80 with S_q a multiple of 128 and S_kv a multiple of 64 run on the tcgen05/TMEM kernel (q, k, v read
 * in place through TMA); every other shape runs the register-resident mma.sync kernel.  workspace / workspace_bytes are
 * kept for ABI stability and ignored (b200sd_attention_workspace_bytes returns 0): no scratch is needed any more.
 * Replaces CrossAttention._attention (baddbmm + softmax + bmm; SURVEY.md K4). */
size_t b200sd_attention_workspace_bytes(int batch, int heads, int Skv, int d);
int b200sd_attention(const void* q, const void* k, const void* v, void* out, int batch, int heads, int Sq, int Skv,
                     int d, int ldq, int ldk, int ldv, int ldo, float scale, void* workspace, size_t workspace_bytes,
                     b200sd_stream_t stream);

/* Same as b200sd_attention, additionally writing lse[batch][heads][Sq] (fp32): the log2-domain
 * log-sum-exp of the scaled scores, log2(sum_j exp(scale q.k_j)), which b200sd_attention_bwd needs.
 * lse may be NULL. */
int b200sd_attention_lse(const void* q, const void* k, const void* v, void* out, float* lse, int batch, int heads, int Sq,
                         int Skv, int d, int ldq, int ldk, int ldv, int ldo, float scale, void* workspace,
                         size_t workspace_bytes, b200sd_stream_t stream);

/* Backward of the fused attention (autograd through CrossAttention._attention; SURVEY.md A5/A9):
 *   dV = P^T dO;  dS = P o (dO V^T - rowsum(dO o O)) * scale;  dQ = dS K;  dK = dS^T Q
 * with P recomputed from lse (never materialised).  q/k/v/out/dout and dq/dk/dv are bf16 row-major
 * buffers addressed like b200sd_attention (head h at columns [h*d, (h+1)*d), own leading dims), so the
 * gradients can be written straight into the column slices of a fused [M, 3C] / [M, 2C] buffer.
 * workspace: b200sd_attention_bwd_workspace_bytes (delta). Deterministic (no atomics). */
size_t b200sd_attention_bwd_workspace_bytes(int batch, int heads, int Sq);
int b200sd_attention_bwd(const void* q, const void* k, const void* v, const void* out, const void* dout,
                         const float* lse, void* dq, void* dk, void* dv, int batch, int heads, int Sq, int Skv, int d,
                         int ldq, int ldk, int ldv, int ldo, int lddo, int lddq, int lddk, int lddv, float scale,
                         void* workspace, size_t workspace_bytes, b200sd_stream_t stream);

/* ---- CLIP text encoder (SURVEY.md 8f N3): the non-GEMM kernels of transformers' CLIPTextModel forward / backward ----------
 * Reference call sites: finetune_sd.py:322-324 (load), 375-379 (train), 477 (`text_encoder(batch["input_ids"])[0]`).
 * The linears of the 12 layers run on b200sd_gemm / _dgrad / _wgrad, LayerNorm 1/2 on b200sd_layernorm(_bwd). */

/* x[b*S + s][:] = tok[ids[b][s]][:] + pos[s][:]   (ids int64 [batch][S]; tok fp32 [vocab][C]; pos fp32 [S][C]; x fp32). */
int b200sd_clip_embed(const int64_t* ids, const float* tok, const float* pos, float* out, int batch, int S, int C, int vocab,
                      b200sd_stream_t stream);
/* dtok[ids[b][s]] += dx[b][s] (fp32 atomics: a token may repeat), dpos[s] += sum_b dx[b][s] (fixed order). */
int b200sd_clip_embed_bwd(const int64_t* ids, const float* dx, float* dtok, float* dpos, int batch, int S, int C, int vocab,
                          b200sd_stream_t stream);
/* quick-GELU (CLIP's hidden_act): out = u * sigmoid(1.702 u);  du = dg * d/du of that.  bf16, n % 8 == 0. */
int b200sd_quick_gelu_fwd(const void* u, void* out, int64_t n, b200sd_stream_t stream);
int b200sd_quick_gelu_bwd(const void* u, const void* dg, void* du, int64_t n, b200sd_stream_t stream);
/* LayerNorm fp32 [rows, C] -> fp32 (CLIP's final_layer_norm: the text context keeps fp32). */
int b200sd_layernorm_f32out(const float* x, const float* gamma, const float* beta, float* out, int rows, int C, float eps,
                            b200sd_stream_t stream);
/* Causal multi-head attention over S <= 96 tokens, head dim d <= 64 (d % 8 == 0): one CTA per (prompt, head), Q/K/V/P of
 * the head in shared memory.  qkv bf16 [batch*S][ld] with q / k / v of head h at columns {q,k,v}_off + h*d;
 * out bf16 [batch*S][ldo] at column h*d.  out = softmax_causal(scale * q k^T) v. */
int b200sd_causal_attention(const void* qkv, void* out, int batch, int heads, int S, int d, int ld, int ldo, int q_off,
                            int k_off, int v_off, float scale, b200sd_stream_t stream);
/* Backward of b200sd_causal_attention (probabilities recomputed; deterministic): dqkv bf16 [batch*S][ldd], same column
 * layout as qkv; dout bf16 [batch*S][lddo]. */
int b200sd_causal_attention_bwd(const void* qkv, const void* dout, void* dqkv, int batch, int heads, int S, int d, int ld,
                                int lddo, int ldd, int q_off, int k_off, int v_off, float scale, b200sd_stream_t stream);

/* ---- AutoencoderKL (SURVEY.md 8f N1): what the VAE needs beyond the UNet's kernels -------------------------------------
 * Reference call sites: finetune_sd.py:325-327 (load), 460-462 (`vae.encode(pixel_values).latent_dist.sample() * 0.18215`),
 * and `vae.decode(latents / 0.18215)` inside every pipeline(...) call (inference.py:175-176, 342-351).
 * b200sd_gemm's conv3x3 accepts image rows wider than one 128-pixel tile (W % 128 == 0) for the 256 / 512-pixel levels. */

/* b200sd_im2col_s2 with the padding as an argument: pad = 1 is the UNet's Downsample2D, pad = 0 the VAE encoder's
 * `F.pad(x, (0, 1, 0, 1))` + stride-2 conv (taps beyond the right / bottom edge read zero). */
int b200sd_im2col_s2_pad(const void* x, void* out, int batch, int H, int W, int C, int in_dtype, int pad,
                         b200sd_stream_t stream);
/* out[r][0..L) = softmax(scale * x[r][0..L))  fp32 [rows][ldx] -> bf16 [rows][ldo]: the probabilities of the mid block's
 * single-head attention between its two GEMMs (scores = q k^T as b200sd_gemm, out = P v as b200sd_gemm_dgrad). */
int b200sd_softmax_rows(const float* x, void* out_bf16, int rows, int L, int ldx, int ldo, float scale, b200sd_stream_t stream);
/* 1x1 convolution over <= 8 channels, NCHW fp32 -> NCHW fp32 (post_quant_conv; w [Cout][Cin]). */
int b200sd_conv1x1_small(const float* x_nchw, const float* w, const float* bias, float* out_nchw, int batch, int Cin, int Cout,
                         int hw, b200sd_stream_t stream);
/* DiagonalGaussianDistribution: moments NCHW [batch][2C][hw] = [mean | logvar];
 * out = (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise) * out_scale; noise == NULL gives the mode. */
int b200sd_gaussian_sample(const float* moments, const float* noise, float* out, int batch, int C, int hw, float out_scale,
                           b200sd_stream_t stream);

/* ---- non-GEMM kernels of the backward pass (SURVEY.md A9) ----------------------------------- */

/* Gradient prep: optional bf16 copy of a [rows, N] (pitch ld) gradient (the tensor-core operand of
 * dgrad / wgrad) and optional column sums ACCUMULATED into colsum (the bias gradient).  With
 * rows_per_image > 0 the sums are kept per image: colsum[image * ldcs + n] (time-embedding gradient). */
int b200sd_grad_prep(const void* in, int in_dtype, void* out_bf16, float* colsum, int rows, int N, int ld,
                     int rows_per_image, int ldcs, b200sd_stream_t stream);

/* Backward of b200sd_groupnorm_silu.  dy: bf16 [rows, C0+C1] gradient of the (activated) output.
 * out0 [rows, C0] / out1 [rows, C1] (out_dtype) receive dx (+ add_src, an optional fp32 [rows, C0+C1]
 * addend: the residual path), overwritten or accumulated per the accumulate flags.  dgamma / dbeta
 * (fp32 [C0+C1]) are ACCUMULATED; pass NULL for both when the parameters are frozen.
 * mean_rstd: the forward's stats_out (fast path: one vectorised pass for the per-channel sums), or NULL (the group
 * statistics are recomputed).  workspace: float[b200sd_groupnorm_bwd_workspace_floats(batch)] of plain scratch.
 * dx is bit-reproducible (per-slab partial sums folded in a fixed order); dgamma / dbeta are fp32 atomics. */
int b200sd_groupnorm_bwd_workspace_floats(int batch);
int b200sd_groupnorm_silu_bwd(const void* x0, const void* x1, int C0, int C1, int in_dtype, const float* gamma,
                              const float* beta, const void* dy, const float* add_src, void* out0, void* out1,
                              int out_dtype, int accumulate0, int accumulate1, float* dgamma, float* dbeta,
                              const float* mean_rstd, float* workspace, int batch, int hw, int groups, float eps, int silu,
                              b200sd_stream_t stream);

/* Backward of b200sd_layernorm: dres[rows, C] (fp32) += dx;  dgamma / dbeta accumulated (or both NULL). */
int b200sd_layernorm_bwd(const void* x, int in_dtype, const float* gamma, const void* dy, float* dres, float* dgamma,
                         float* dbeta, int rows, int C, float eps, b200sd_stream_t stream);

/* GEGLU of the training path (pre-activation kept): u bf16 [rows, 2*C_half] = [values | gates];
 * out[rows, C_half] = values * gelu_erf(gates);  du = d/du of that given dff [rows, C_half]. */
int b200sd_geglu_fwd(const void* u, void* out, int64_t rows, int C_half, b200sd_stream_t stream);
int b200sd_geglu_bwd(const void* u, const void* dff, void* du, int64_t rows, int C_half, b200sd_stream_t stream);

/* Transposes of the resamplers: dy bf16 (batch,2H,2W,C) -> dx fp32 (batch,H,W,C) (sum of 2x2 blocks);
 * dcol bf16 [batch*(H/2)*(W/2)][9*C] -> dx fp32 (batch,H,W,C).  accumulate != 0: dx += . */
int b200sd_upsample2x_bwd(const void* dy, float* dx, int batch, int H, int W, int C, int accumulate, b200sd_stream_t stream);
int b200sd_col2im_s2(const void* dcol, float* dx, int batch, int H, int W, int C, int accumulate, b200sd_stream_t stream);

/* Backward of b200sd_conv_out: dx_nhwc (bf16 [batch*H*W, Cin]) = data gradient; when dw != NULL also
 * dw[Cout][9][Cin] += weight gradient (needs x_nhwc, the forward input) and dbias[Cout] += sum(dout). */
int b200sd_conv_out_bwd(const float* dout_nchw, const void* x_nhwc, const float* w, void* dx_nhwc, float* dw,
                        float* dbias, int batch, int Cin, int Cout, int H, int W, b200sd_stream_t stream);
/* Weight gradient of b200sd_conv_in: dw[Cout][9][Cin] += sum_p dy[p, co] x[b, ci, p + d(tap)]. */
int b200sd_conv_in_wgrad(const void* dy_nhwc, int dy_dtype, const float* x_nchw, float* dw, int batch, int Cin, int Cout,
                         int H, int W, b200sd_stream_t stream);

/* out_bf16[i] = act(in[i]) (act = SiLU when silu != 0);  grad[i] *= silu'(pre[i])  (time-embedding MLP backward) */
int b200sd_cast_act(const float* in, void* out_bf16, int64_t n, int silu, b200sd_stream_t stream);
int b200sd_silu_bwd_mul(const float* pre, float* grad, int64_t n, b200sd_stream_t stream);

/* ---- fp32-accuracy path (north_star: "the fp32 path within 1e-4") ------------------------------
 * The tensor cores stay bf16: an fp32 operand x travels as (hi, lo) = (bf16(x), bf16(x - hi)) and a product is
 * evaluated as A_hi B_hi + A_lo B_hi + A_hi B_lo with fp32 accumulation -- two b200sd_gemm calls:
 * [A_hi | A_lo] x [B_hi | B_hi]^T (a0 / a1 K-concat), then A_hi x B_lo^T added through the fp32 residual input. */
int b200sd_split_hi_lo(const float* x, void* hi_bf16, void* lo_bf16, int64_t n, b200sd_stream_t stream);
/* GroupNorm / LayerNorm that also emit the lo halves (out_lo / raw_lo may be NULL; stats_out as in _stats). */
int b200sd_groupnorm_silu_split(const void* x0, const void* x1, int C0, int C1, const float* gamma, const float* beta,
                                void* out, void* out_lo, void* raw_out, void* raw_lo, float* stats_ws, float* stats_out,
                                int batch, int hw, int groups, float eps, int silu, int in_dtype, b200sd_stream_t stream);
int b200sd_layernorm_split(const void* x, const float* gamma, const float* beta, void* out, void* out_lo, int rows, int C,
                           float eps, int in_dtype, b200sd_stream_t stream);
/* u fp32 [rows, 2*C_half] = [values | gates] -> (hi, lo) of values * gelu_erf(gates), each bf16 [rows, C_half] */
int b200sd_geglu_f32(const float* u, void* hi_bf16, void* lo_bf16, int64_t rows, int C_half, b200sd_stream_t stream);
/* fp32 flash attention on the CUDA cores (online softmax with expf, no score matrix in HBM); q is pre-multiplied by
 * scale inside; same addressing as b200sd_attention but fp32 buffers; d in {8,16,32,40,64,80,128,160}. */
int b200sd_attention_f32(const float* q, const float* k, const float* v, float* out, int batch, int heads, int Sq, int Skv,
                         int d, int ldq, int ldk, int ldv, int ldo, float scale, b200sd_stream_t stream);
/* b200sd_small_linear with fp32 weights (time-embedding MLP and time_emb_proj heads of the fp32 path) */
int b200sd_small_linear_f32(const float* in, const float* w, const float* bias, float* out, int batch, int N, int K,
                            int silu_in, int silu_out, b200sd_stream_t stream);

/* ---- optimizer step over the flat kernel-layout buffers (finetune_sd.py:407-420, 569-570) ------ */
/* out_bf16[i] = in[i] for n (multiple of 8) elements: fp32 master weights -> bf16 tensor-core copy. */
int b200sd_cast_flat(const float* in, void* out_bf16, int64_t n, b200sd_stream_t stream);
/* torch.optim.AdamW semantics (decoupled weight decay, bias correction with `step` >= 1) over n
 * (multiple of 4) parameters, fused with: gradient scaling (grad_scale = 1 / world averages a SUM
 * allreduce), the bf16 re-cast of the updated weights, and optional zeroing of grad for the next step.
 * HBM-bound: 16 B read + 14 B (18 B with zero_grad) written per parameter. */
int b200sd_adamw_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, void* weights_bf16, int64_t n,
                      float lr, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                      int zero_grad, b200sd_stream_t stream);

/* bnb.optim.AdamW8bit semantics -- the reference's default optimizer (finetune_sd.py:300 use_8bit_adam=True, :407-420
 * `bnb.optim.AdamW8bit(params, lr, weight_decay, min_8bit_size=16384)`; bitsandbytes 0.35.4, un-vendored) -- over the n (multiple
 * of 64) parameters of a flat buffer: both Adam moments are stored as 1-byte codes of a 256-entry code book (`qmap1` signed,
 * `qmap2` unsigned: bitsandbytes' "dynamic" maps, sorted ascending) times one fp32 absmax per block of 2048 values
 * (`absmax1/2`: ceil(n / 2048) floats).  `chunk_mode` (n / 64 ints, or NULL = every value 8-bit) says, per 64-value chunk of the
 * flat buffer: -1 = 8-bit moments, -2 = frozen / padding (nothing read or written), k >= 0 = fp32 moments at
 * small_exp_avg[k ..] / small_exp_avg_sq[k ..] (tensors below min_8bit_size).  Update (bitsandbytes' order):
 * m = b1 m + (1-b1) g; v = b2 v + (1-b2) g g; p += -lr sqrt(1-b2^t)/(1-b1^t) * m / (sqrt(v) + sqrt(1-b2^t) eps); p *= 1 - lr wd;
 * re-quantise m / max|m|, v / max|v| to the nearest code.  Fused like b200sd_adamw_step: grad_scale, bf16 re-cast of the weights,
 * optional zeroing of grad.  HBM-bound: 10 B read + 8 B (12 B with zero_grad) written per parameter. */
int b200sd_adamw8bit_step(float* param, float* grad, uint8_t* state1, uint8_t* state2, float* absmax1, float* absmax2,
                          const float* qmap1, const float* qmap2, const int32_t* chunk_mode, float* small_exp_avg,
                          float* small_exp_avg_sq, void* weights_bf16, int64_t n, float lr, float beta1, float beta2, float eps,
                          float weight_decay, int step, float grad_scale, int zero_grad, b200sd_stream_t stream);

/* nearest x2 upsample NHWC bf16: (batch,H,W,C) -> (batch,2H,2W,C)  (Upsample2D's F.interpolate) */
int b200sd_upsample2x(const void* x, void* out, int batch, int H, int W, int C, int in_dtype, b200sd_stream_t stream);
/* im2col for the three stride-2 Downsample2D convs: NHWC (batch,H,W,C) -> [batch*(H/2)*(W/2)][9*C] */
int b200sd_im2col_s2(const void* x, void* out, int batch, int H, int W, int C, int in_dtype, b200sd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200SD_H_ */
