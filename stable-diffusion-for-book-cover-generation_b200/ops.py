"""Thin torch-tensor wrappers over the C ABI (include/b200sd.h).  Tensors are torch-owned device
memory; every call goes to libb200sd.so on torch's current CUDA stream.  No CPU / eager fallback:
a non-CUDA tensor is an error."""
from __future__ import annotations

import ctypes as C

import torch

from ._lib import DgradArgs, GemmArgs, WgradArgs, B200SDError, check, lib

F32, BF16 = 0, 1
EPI_LINEAR, EPI_GEGLU = 0, 1


def _up16(*ts):
    """fp16 tensors (the reference builds every pipeline with torch_dtype=torch.float16: inference.py:406, 425; utils.py:189,
    249) are upcast to fp32 at the Python boundary -- the kernels compute in fp32 either way -- and the caller casts the
    result back.  Returns (tensors..., had_fp16)."""
    had = any(t is not None and t.dtype == torch.float16 for t in ts)
    return tuple(t.float() if (t is not None and t.dtype == torch.float16) else t for t in ts) + (had,)


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise B200SDError(f"unsupported dtype {t.dtype} (float32 / bfloat16 only)")


def _chk(*ts):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise B200SDError("b200sd ops need CUDA tensors (there is no CPU fallback)")
        if not t.is_contiguous():
            raise B200SDError("b200sd ops need contiguous tensors")


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


_ws_cache: dict = {}
_ws_retired: list = []


def _workspace(key, nbytes, device, zero=True):
    k = (key, device.index if device.index is not None else torch.cuda.current_device())
    t = _ws_cache.get(k)
    if t is None or t.numel() < nbytes:
        if t is not None:
            _ws_retired.append(t)   # a captured CUDA graph may still hold its address: outgrown scratch is kept, never freed
        t = (torch.zeros if zero else torch.empty)(nbytes, dtype=torch.uint8, device=device)
        _ws_cache[k] = t
    return t


def attention_workspace_bytes(batch, heads, Skv, d) -> int:
    return int(lib().b200sd_attention_workspace_bytes(batch, heads, Skv, d))


def attention_bwd_workspace_bytes(batch, heads, Sq) -> int:
    return int(lib().b200sd_attention_bwd_workspace_bytes(batch, heads, Sq))


def launch_count() -> int:
    return int(lib().b200sd_launch_count())


# ---------------------------------------------------------------------------------------------
# scheduler / loss elementwise
# ---------------------------------------------------------------------------------------------
def cfg_ddim_step(eps_u, eps_c, x, guidance, sa_t, sb_t, sa_p, sb_p, out=None):
    """DDIM update at eta = 0: sa_p x0 + sb_p eps, x0 = (x - sb_t eps) / sa_t"""
    return cfg_ancestral_step(eps_u, eps_c, x, None, guidance, sa_t, sb_t, sa_p, 0.0, sb_p, 0.0, False, out=out)


def cfg_ancestral_step(eps_u, eps_c, x, noise, guidance, sa_t, sb_t, c_x0, c_x, c_e, c_z, clip, out=None):
    """DDPM / DDIM update: c_x0 x0 + c_x x + c_e eps + c_z noise, x0 = (x - sb_t eps) / sa_t (clamped if clip).
    noise: fp32 with x's size, or None for no noise term."""
    eps_u, eps_c, x, half = _up16(eps_u, eps_c, x)
    if half:
        r = cfg_ancestral_step(eps_u.contiguous(), None if eps_c is None else eps_c.contiguous(), x.contiguous(), noise, guidance,
                               sa_t, sb_t, c_x0, c_x, c_e, c_z, clip).half()
        return r if out is None else out.copy_(r)
    _chk(eps_u, eps_c, x, noise, out)
    if out is None:
        out = torch.empty_like(x)
    if eps_c is not None and eps_c.shape != eps_u.shape:
        raise ValueError("eps_u / eps_c shape mismatch")
    if eps_u.numel() != x.numel():
        raise ValueError(f"model_output {tuple(eps_u.shape)} and sample {tuple(x.shape)} sizes differ")
    if noise is not None and (noise.dtype != torch.float32 or noise.numel() != x.numel()):
        raise ValueError(f"noise must be float32 with {x.numel()} elements")
    check(lib().b200sd_cfg_ancestral_step(_p(eps_u), _p(eps_c), _p(x), _p(noise), _p(out), x.numel(), float(guidance),
                                          float(sa_t), float(sb_t), float(c_x0), float(c_x), float(c_e), float(c_z), int(bool(clip)),
                                          _dt(eps_u), _dt(x), _stream()), "cfg_ancestral_step")
    return out


def cfg_plms_step(eps_u, eps_c, x, hist, weights, guidance, cx, ce, out=None, eps_out=None):
    eps_u, eps_c, x, half = _up16(eps_u, eps_c, x)
    if half:
        # the eps history (eps_out / hist) stays fp32: it never leaves the scheduler
        r = cfg_plms_step(eps_u.contiguous(), None if eps_c is None else eps_c.contiguous(), x.contiguous(), hist, weights, guidance,
                          cx, ce, eps_out=eps_out).half()
        return r if out is None else out.copy_(r)
    _chk(eps_u, eps_c, x, out, eps_out, *hist)
    if out is None:
        out = torch.empty_like(x)
    if eps_u.numel() != x.numel():
        raise ValueError(f"model_output {tuple(eps_u.shape)} and sample {tuple(x.shape)} sizes differ")
    w = (C.c_float * 5)(*([float(v) for v in weights] + [0.0] * (5 - len(weights))))
    hp = [_p(h) for h in hist] + [None] * (4 - len(hist))
    check(lib().b200sd_cfg_plms_step(_p(eps_u), _p(eps_c), _p(x), _p(out), _p(eps_out), hp[0], hp[1], hp[2], hp[3],
                                     len(hist), w, x.numel(), float(guidance), float(cx), float(ce), _dt(eps_u), _dt(x),
                                     _stream()), "cfg_plms_step")
    return out


def sampler_advance(t_table, cursor, in_t):
    """in_t[:] = t_table[cursor[0]]; cursor[0] += 1 (device-side step index of a captured denoising loop)"""
    check(lib().b200sd_sampler_advance(_p(t_table), t_table.numel(), _p(cursor), _p(in_t), in_t.numel(), _stream()),
          "sampler_advance")


def cfg_ancestral_step_table(eps_u, eps_c, x, noise, guidance, coef_table, cursor):
    """cfg_ancestral_step() with row coef_table[cursor[1]] (sa_t sb_t c_x0 c_x c_e c_z noise_row clip) and z = noise[noise_row]
    (fp32 tensors); x is updated in place"""
    check(lib().b200sd_cfg_ancestral_step_table(_p(eps_u), _p(eps_c), _p(x), _p(noise), x.numel(), float(guidance),
                                                _p(coef_table), _p(cursor), _stream()), "cfg_ancestral_step_table")


def cfg_plms_step_table(eps_u, eps_c, x, saved, ring, guidance, coef_table, cursor):
    """cfg_plms_step() with weights, eps-ring slots and saved-sample flags read from coef_table[cursor[0]]; x is updated in place"""
    check(lib().b200sd_cfg_plms_step_table(_p(eps_u), _p(eps_c), _p(x), _p(saved), _p(ring), x.numel(), float(guidance),
                                           _p(coef_table), _p(cursor), _stream()), "cfg_plms_step_table")


def add_noise(x0, noise, timesteps, sa_table, sb_table, out=None):
    x0, noise, half = _up16(x0, noise)
    if half:
        r = add_noise(x0.contiguous(), noise.contiguous(), timesteps, sa_table, sb_table).half()
        return r if out is None else out.copy_(r)
    _chk(x0, noise, timesteps, sa_table, sb_table, out)
    if x0.shape != noise.shape:
        raise ValueError("original_samples / noise shape mismatch")
    if timesteps.dtype != torch.int64 or timesteps.numel() != x0.shape[0]:
        raise ValueError("timesteps must be int64 of shape (batch,)")
    if noise.dtype != x0.dtype:
        noise = noise.to(x0.dtype)
    if out is None:
        out = torch.empty_like(x0)
    B = x0.shape[0]
    check(lib().b200sd_add_noise(_p(x0), _p(noise), _p(timesteps), _p(sa_table), _p(sb_table), _p(out), B,
                                 x0.numel() // max(B, 1), sa_table.numel(), _dt(x0), _stream()), "add_noise")
    return out


def _blend_args(x, x0, noise, mask, sa_table, sb_table):
    _chk(x, x0, noise, mask, sa_table, sb_table)
    for t in (x, x0, noise, mask, sa_table, sb_table):
        if t.dtype != torch.float32:
            raise B200SDError("inpaint_blend is fp32")
    if not x.shape == x0.shape == noise.shape == mask.shape:
        raise ValueError("inpaint_blend: x, x0, noise and mask must have the same shape (expand the mask first)")
    return _p(x), _p(x0), _p(noise), _p(mask), x.numel()


def inpaint_blend(x, x0, noise, mask, timestep, sa_table, sb_table):
    """x <- mask (sa[t] x0 + sb[t] noise) + (1 - mask) x in place (legacy inpainting's masking step at loop timestep t)"""
    args = _blend_args(x, x0, noise, mask, sa_table, sb_table)
    check(lib().b200sd_inpaint_blend(*args, int(timestep), _p(sa_table), _p(sb_table), sa_table.numel(), _stream()),
          "inpaint_blend")
    return x


def inpaint_blend_table(x, x0, noise, mask, t_table, cursor, sa_table, sb_table):
    """inpaint_blend() at t = t_table[cursor[1]], read on the device (the captured sampler's step)"""
    args = _blend_args(x, x0, noise, mask, sa_table, sb_table)
    check(lib().b200sd_inpaint_blend_table(*args, _p(t_table), _p(cursor), _p(sa_table), _p(sb_table), sa_table.numel(),
                                           _stream()), "inpaint_blend_table")
    return x


def cfg_sigma_step(eps_u, eps_c, x, guidance, sigma, coefs, hist=(), noise=None, sigma_up=0.0, out=None, d_out=None):
    """Step of the sigma-space schedulers (LMS, Euler, Euler-a): d = (x - (x - sigma eps)) / sigma, eps the CFG combine;
    out = x + sum(coefs[k] * [d, *hist][k]) (+ sigma_up noise).  hist: up to 3 earlier derivatives, newest first.  eps fp32 or
    bf16; x, hist, noise, out and d_out (receives d) fp32."""
    _chk(eps_u, eps_c, x, noise, out, d_out, *hist)
    if len(coefs) != len(hist) + 1 or len(hist) > 3:
        raise ValueError(f"cfg_sigma_step: {len(coefs)} coefficients for {len(hist)} history terms (up to 3)")
    for t in (x, noise, out, d_out, *hist):
        if t is not None and (t.dtype != torch.float32 or t.numel() != x.numel()):
            raise ValueError(f"cfg_sigma_step: x, noise, history, out and d_out must be float32 with {x.numel()} elements")
    if eps_c is not None and eps_c.shape != eps_u.shape:
        raise ValueError("eps_u / eps_c shape mismatch")
    if eps_u.numel() != x.numel():
        raise ValueError(f"model_output {tuple(eps_u.shape)} and sample {tuple(x.shape)} sizes differ")
    if out is None:
        out = torch.empty_like(x)
    c = [float(v) for v in coefs] + [0.0] * (4 - len(coefs))
    hp = [_p(h) for h in hist] + [None] * (3 - len(hist))
    check(lib().b200sd_cfg_sigma_step(_p(eps_u), _p(eps_c), _p(x), _p(noise), _p(out), _p(d_out), hp[0], hp[1], hp[2],
                                      x.numel(), float(guidance), float(sigma), *c, float(sigma_up), _dt(eps_u), _stream()),
          "cfg_sigma_step")
    return out


def cfg_sigma_step_table(eps_u, eps_c, x, ring, noise, guidance, coef_table, cursor):
    """cfg_sigma_step() with row coef_table[cursor[1]] (sigma | c0..c3 | h1 h2 h3 | out_slot | noise_row | sigma_up | in_div):
    history from / derivative to the 4-slot `ring`, z = noise[noise_row] (fp32 tensors); x is updated in place"""
    check(lib().b200sd_cfg_sigma_step_table(_p(eps_u), _p(eps_c), _p(x), _p(ring), _p(noise), x.numel(), float(guidance),
                                            _p(coef_table), _p(cursor), _stream()), "cfg_sigma_step_table")


def sampler_scale_input(x, x2, coef_table, cursor):
    """x2[:B] = x2[B:] = x / in_div of row coef_table[cursor[1]] (fp32): the scaled UNet input of a sigma-space captured step"""
    if x2.numel() != 2 * x.numel():
        raise ValueError("sampler_scale_input: x2 must hold two copies of x")
    check(lib().b200sd_sampler_scale_input(_p(x), _p(x2), x.numel(), _p(coef_table), _p(cursor), _stream()),
          "sampler_scale_input")


def sampler_inpaint_input(latents, cond, x2, coef_table=None, cursor=None):
    """x2[n] = [latents[n mod B] | cond[n mod B]] for n in [0, 2B), divided by in_div of row coef_table[cursor[1]] when a table is
    given (fp32 NCHW): the input of a captured step of the 9-channel inpainting UNet, concatenated then scaled as in 0.7.2"""
    _chk(latents, cond, x2, coef_table, cursor)
    B, c_lat, h, w = latents.shape
    c_cond = cond.shape[1]
    if tuple(cond.shape) != (B, c_cond, h, w) or tuple(x2.shape) != (2 * B, c_lat + c_cond, h, w):
        raise ValueError(f"sampler_inpaint_input: latents {tuple(latents.shape)}, cond {tuple(cond.shape)} and x2 {tuple(x2.shape)} "
                         "do not fit together")
    if any(t is not None and t.dtype != torch.float32 for t in (latents, cond, x2, coef_table)):
        raise B200SDError("sampler_inpaint_input is fp32")
    if (coef_table is None) != (cursor is None):
        raise ValueError("sampler_inpaint_input: pass coef_table and cursor together")
    check(lib().b200sd_sampler_inpaint_input(_p(latents), _p(cond), _p(x2), B, c_lat, c_cond, h * w, _p(coef_table), _p(cursor),
                                             _stream()), "sampler_inpaint_input")
    return x2


def mse_loss_fwd(pred, target):
    _chk(pred, target)
    if pred.shape != target.shape:
        raise ValueError("pred / target shape mismatch")
    ws = _workspace("mse", lib().b200sd_mse_workspace_floats() * 4, pred.device)
    out = torch.empty(1, dtype=torch.float32, device=pred.device)
    check(lib().b200sd_mse_loss_fwd(_p(pred), _p(target), _p(out), _p(ws), pred.numel(), _dt(pred), _dt(target),
                                    _stream()), "mse_loss_fwd")
    return out


def mse_loss_bwd(pred, target, grad_loss):
    _chk(pred, target, grad_loss)
    g = torch.empty_like(pred)
    gl = grad_loss.reshape(1).to(torch.float32)
    check(lib().b200sd_mse_loss_bwd(_p(pred), _p(target), _p(gl), _p(g), pred.numel(), _dt(pred), _dt(target),
                                    _stream()), "mse_loss_bwd")
    return g


class _MSELoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target):
        ctx.pred_dtype = pred.dtype
        pred, target, _ = _up16(pred, target)          # fp16 (autocast / fp16 pipelines): the loss is computed in fp32 as F.mse_loss under autocast
        ctx.save_for_backward(pred, target)
        return mse_loss_fwd(pred.contiguous(), target.contiguous()).reshape(())

    @staticmethod
    def backward(ctx, grad):
        pred, target = ctx.saved_tensors
        return mse_loss_bwd(pred.contiguous(), target.contiguous(), grad.contiguous().float()).to(ctx.pred_dtype), None


def mse_loss(pred, target):
    """== F.mse_loss(pred, target, reduction="none").mean([1,2,3]).mean() (finetune_sd.py:483-484)."""
    return _MSELoss.apply(pred, target)


# ---------------------------------------------------------------------------------------------
# UNet building blocks
# ---------------------------------------------------------------------------------------------
def timestep_embedding(t_f32, dim, out=None):
    _chk(t_f32, out)
    B = t_f32.numel()
    if out is None:
        out = torch.empty(B, dim, dtype=torch.float32, device=t_f32.device)
    check(lib().b200sd_timestep_embedding(_p(t_f32), _p(out), B, dim, _stream()), "timestep_embedding")
    return out


def small_linear(x, w_bf16, bias, silu_in=False, silu_out=False, out=None):
    _chk(x, w_bf16, bias, out)
    B, K = x.shape
    N = w_bf16.shape[0]
    if out is None:
        out = torch.empty(B, N, dtype=torch.float32, device=x.device)
    check(lib().b200sd_small_linear(_p(x), _p(w_bf16), _p(bias), _p(out), B, N, K, int(silu_in), int(silu_out),
                                    _stream()), "small_linear")
    return out


def gemm_workspace(device):
    """Split-K scratch of the GEMM kernels (partial tiles + self-resetting counters, zeroed once).  One buffer per (device, stream):
    launches that share it must be stream-ordered."""
    return _workspace(("gemm", _stream()), max(16, lib().b200sd_gemm_workspace_bytes()), device)


def gemm(a0, w, out, *, a1=None, bias=None, rowbias=None, residual=None, conv=None, rows_per_image=0,
         epilogue=EPI_LINEAR, block_n=0, split_k=0, M=None, ldrb=0, launch=True, pair=0):
    """out[M, N] = [a0 | a1] @ w^T (+bias +rowbias +residual); conv=(batch, H, W) -> 3x3 pad-1 conv (NHWC)."""
    _chk(a0, a1, w, bias, rowbias, residual, out)
    N, K = w.shape
    C0 = a0.shape[-1]
    C1 = a1.shape[-1] if a1 is not None else 0
    if M is None:
        M = a0.numel() // C0
    ws = gemm_workspace(a0.device)
    args = GemmArgs()
    args.a0, args.a1, args.w = _p(a0), _p(a1), _p(w)
    args.bias, args.rowbias, args.residual, args.out = _p(bias), _p(rowbias), _p(residual), _p(out)
    args.M, args.N, args.K, args.C0, args.C1 = M, N, K, C0, C1
    args.lda0, args.lda1 = C0, C1
    args.ldc = out.shape[-1]
    args.ldr = residual.shape[-1] if residual is not None else 0
    args.ldrb = ldrb
    if conv is not None:
        args.conv_taps = 9
        args.batch, args.H, args.W = conv
    else:
        args.conv_taps = 1
    args.rows_per_image = rows_per_image
    args.epilogue = epilogue
    args.out_dtype = _dt(out)
    args.residual_dtype = _dt(residual) if residual is not None else BF16
    args.block_n, args.split_k = block_n, split_k
    args.pair = pair
    args.workspace, args.workspace_bytes = _p(ws), ws.numel()
    if not launch:
        return args
    gemm_run(args)
    return out


def gemm_run(args):
    check(lib().b200sd_gemm(C.byref(args), _stream()), "gemm")


_GEMM_PATH_FIELDS = ("kernel", "split_k", "psplit", "pair", "block_n", "m_tiles", "n_tiles", "rows_valid", "tile_n", "tiles_x")
_GEMM_KERNELS = ("tile", "persistent", "persistent-split")


def gemm_path(args) -> dict:
    """The kernel and tiling gemm_run(args) would launch (b200sd_gemm_describe: the launch's own decision, nothing launched).
    kernel is "tile" (one output tile per CTA), "persistent" or "persistent-split" (its K-sliced mode)."""
    f = (C.c_int * len(_GEMM_PATH_FIELDS))()
    check(lib().b200sd_gemm_describe(C.byref(args), f), "gemm_describe")
    d = dict(zip(_GEMM_PATH_FIELDS, f))
    d["kernel"] = _GEMM_KERNELS[d["kernel"]]
    return d


class GnParts:
    """Column statistics a GEMM writes next to its fp32 output (GemmArgs.gn_part) for the GroupNorm that consumes it:
    buf [total_parts][2][N] floats; image b owns partial rows [b * ppi, (b + 1) * ppi)."""
    __slots__ = ("buf", "ppi", "ld")

    def __init__(self, buf, ppi, ld):
        self.buf, self.ppi, self.ld = buf, ppi, ld


def gemm_attach_gn_parts(args, hw, device):
    """Ask the library how a GEMM with `args` would lay out its GroupNorm statistics (hw = output rows per image); when
    the shape is covered, allocate the buffer, point args.gn_part at it and return a GnParts, else return None."""
    ppi, total = C.c_int(0), C.c_int(0)
    check(lib().b200sd_gemm_gn_layout(C.byref(args), int(hw), C.byref(ppi), C.byref(total)), "gemm_gn_layout")
    if ppi.value <= 0:
        return None
    buf = torch.zeros(total.value * 2 * args.N, dtype=torch.float32, device=device)
    args.gn_part = buf.data_ptr()
    return GnParts(buf, ppi.value, args.N)


def groupnorm_silu_parts(x0, x1, parts0, parts1, gamma, beta, out, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None,
                         stats_out=None):
    """groupnorm_silu() with the statistics taken from the producers' GnParts (check gn_parts_supported(C) first)."""
    _chk(x0, x1, gamma, beta, out, raw_out, stats_out)
    C0 = x0.shape[-1]
    C1 = x1.shape[-1] if x1 is not None else 0
    rc = lib().b200sd_groupnorm_silu_parts(_p(x0), _p(x1), C0, C1, _p(parts0.buf), parts0.ppi, parts0.ld,
                                           _p(parts1.buf) if parts1 is not None else None, parts1.ppi if parts1 is not None else 0,
                                           parts1.ld if parts1 is not None else 0, _p(gamma), _p(beta), _p(out), _p(raw_out),
                                           _p(stats_out), batch, hw, groups, float(eps), int(silu), _dt(x0), _stream())
    check(rc, "groupnorm_silu_parts")
    return out


def gn_parts_supported(C, groups=32):
    """Channel layouts b200sd_groupnorm_silu_parts covers (mirrors its G / Cg choice; anything else returns an error there)."""
    if C % groups:
        return False
    cpg = C // groups
    G = 1
    while (G * cpg) % 8 != 0 and G < groups:
        G *= 2
    while G * 2 <= groups and groups % (G * 2) == 0 and G * cpg < 32:
        G *= 2
    Cg = G * cpg
    return Cg % 8 == 0 and groups % G == 0 and Cg // 8 <= 512


def gemm_dgrad(dy, w, out, *, residual=None, conv=None, Cin=None, block_n=0, launch=True, pair=0):
    """out[M, Cin] = dy[M, Cout] (*) w  (+ residual): data gradient of gemm(); w is the FORWARD weight
    [Cout][taps*Cin]; conv=(batch, H, W) -> gradient of the 3x3 pad-1 conv."""
    _chk(dy, w, residual, out)
    Cout = w.shape[0]
    taps = 9 if conv is not None else 1
    if Cin is None:
        Cin = w.shape[1] // taps
    a = DgradArgs()
    a.dy, a.w, a.residual, a.out = _p(dy), _p(w), _p(residual), _p(out)
    a.M, a.Cout, a.Cin, a.conv_taps = dy.numel() // dy.shape[-1], Cout, Cin, taps
    if conv is not None:
        a.batch, a.H, a.W = conv
    a.ldy, a.ldc = dy.shape[-1], out.shape[-1]
    a.ldr = residual.shape[-1] if residual is not None else 0
    a.out_dtype = _dt(out)
    a.residual_dtype = _dt(residual) if residual is not None else BF16
    a.block_n = block_n
    a.pair = pair
    if not launch:
        return a
    gemm_dgrad_run(a)
    return out


def gemm_dgrad_run(args):
    check(lib().b200sd_gemm_dgrad(C.byref(args), _stream()), "gemm_dgrad")


def gemm_wgrad(dy, x, dw, *, conv=None, lddw=0, block_n=0, split_k=0, launch=True):
    """dw[Cout][taps*Cin] += dy[rows, Cout]^T (*) x[rows, Cin]  (fp32, accumulated with red.add)."""
    _chk(dy, x, dw)
    if dw.dtype != torch.float32:
        raise B200SDError("gemm_wgrad: dw must be float32")
    a = WgradArgs()
    a.dy, a.x, a.dw = _p(dy), _p(x), _p(dw)
    a.rows, a.Cout, a.Cin = dy.numel() // dy.shape[-1], dy.shape[-1], x.shape[-1]
    a.conv_taps = 9 if conv is not None else 1
    if conv is not None:
        a.batch, a.H, a.W = conv
    a.ldy, a.ldx, a.lddw = dy.shape[-1], x.shape[-1], lddw
    a.block_n, a.split_k = block_n, split_k
    if not launch:
        return a
    gemm_wgrad_run(a)
    return dw


def gemm_wgrad_run(args):
    check(lib().b200sd_gemm_wgrad(C.byref(args), _stream()), "gemm_wgrad")


def geglu_tile(N):
    return int(lib().b200sd_geglu_tile(N))


def conv_in(x_nchw, w_packed, bias, out):
    _chk(x_nchw, w_packed, bias, out)
    B, Cin, H, W = x_nchw.shape
    check(lib().b200sd_conv_in(_p(x_nchw), _p(w_packed), _p(bias), _p(out), B, Cin, w_packed.shape[0], H, W, _dt(out), _stream()),
          "conv_in")
    return out


def conv_out(x_nhwc, w_packed, bias, out_nchw):
    _chk(x_nhwc, w_packed, bias, out_nchw)
    B, Cout, H, W = out_nchw.shape
    check(lib().b200sd_conv_out(_p(x_nhwc), _p(w_packed), _p(bias), _p(out_nchw), B, x_nhwc.shape[-1], Cout, H, W,
                                _stream()), "conv_out")
    return out_nchw


def nhwc_bias_to_nchw(x_f32, bias, out_nchw):
    """out_nchw[b][c][p] = x[b*hw + p][c] + bias[c] (x: fp32 [batch*hw][ld], c < out channels <= 4)."""
    _chk(x_f32, bias, out_nchw)
    B, C, H, W = out_nchw.shape
    check(lib().b200sd_nhwc_bias_to_nchw(_p(x_f32), _p(bias), _p(out_nchw), B, C, H * W, x_f32.shape[-1], _stream()), "nhwc_bias_to_nchw")
    return out_nchw


def groupnorm_silu(x0, x1, gamma, beta, out, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None, stats_out=None):
    _chk(x0, x1, gamma, beta, out, raw_out, stats_out)
    if x1 is not None and x1.dtype != x0.dtype:
        raise B200SDError("groupnorm: both sources must have the same dtype")
    ws = _workspace(("gn", _stream()), lib().b200sd_groupnorm_workspace_floats(batch) * 4, x0.device)
    C0 = x0.shape[-1]
    C1 = x1.shape[-1] if x1 is not None else 0
    check(lib().b200sd_groupnorm_silu_stats(_p(x0), _p(x1), C0, C1, _p(gamma), _p(beta), _p(out), _p(raw_out), _p(ws),
                                            _p(stats_out), batch, hw, groups, float(eps), int(silu), _dt(x0), _stream()),
          "groupnorm_silu")
    return out


def layernorm(x, gamma, beta, out, eps=1e-5):
    _chk(x, gamma, beta, out)
    Cc = x.shape[-1]
    check(lib().b200sd_layernorm(_p(x), _p(gamma), _p(beta), _p(out), x.numel() // Cc, Cc, float(eps), _dt(x), _stream()),
          "layernorm")
    return out


def attention(q, k, v, out, batch, heads, Sq, Skv, d, scale, ldq=None, ldk=None, ldv=None, ldo=None,
              q_off=0, k_off=0, v_off=0, ws=None):
    """q/k/v may be column slices of wider row-major buffers: pass the buffer plus an element offset."""
    _chk(q, k, v, out)
    es = 2
    if ws is None:
        ws = _workspace("attn", lib().b200sd_attention_workspace_bytes(batch, heads, Skv, d) + 128, q.device, zero=False)
    check(lib().b200sd_attention(q.data_ptr() + q_off * es, k.data_ptr() + k_off * es, v.data_ptr() + v_off * es,
                                 _p(out), batch, heads, Sq, Skv, d, ldq or q.shape[-1], ldk or k.shape[-1],
                                 ldv or v.shape[-1], ldo or out.shape[-1], float(scale), _p(ws), ws.numel(), _stream()),
          "attention")
    return out


def upsample2x(x, out, batch, H, W):
    _chk(x, out)
    check(lib().b200sd_upsample2x(_p(x), _p(out), batch, H, W, x.shape[-1], _dt(x), _stream()), "upsample2x")
    return out


def im2col_s2(x, out, batch, H, W, pad=1):
    _chk(x, out)
    check(lib().b200sd_im2col_s2_pad(_p(x), _p(out), batch, H, W, x.shape[-1], _dt(x), int(pad), _stream()), "im2col_s2")
    return out


# ---------------------------------------------------------------------------------------------
# backward-pass kernels (SURVEY.md row A9)
# ---------------------------------------------------------------------------------------------
def attention_lse(q, k, v, out, lse, batch, heads, Sq, Skv, d, scale, ldq=None, ldk=None, ldv=None, ldo=None,
                  q_off=0, k_off=0, v_off=0, ws=None):
    """attention() that also writes lse[batch, heads, Sq] (log2-domain log-sum-exp) for attention_bwd()."""
    _chk(q, k, v, out, lse)
    if ws is None:
        ws = _workspace("attn", lib().b200sd_attention_workspace_bytes(batch, heads, Skv, d) + 128, q.device, zero=False)
    check(lib().b200sd_attention_lse(q.data_ptr() + q_off * 2, k.data_ptr() + k_off * 2, v.data_ptr() + v_off * 2,
                                     _p(out), _p(lse), batch, heads, Sq, Skv, d, ldq or q.shape[-1], ldk or k.shape[-1],
                                     ldv or v.shape[-1], ldo or out.shape[-1], float(scale), _p(ws), ws.numel(),
                                     _stream()), "attention_lse")
    return out


def attention_bwd(q, k, v, out, dout, lse, dq, dk, dv, batch, heads, Sq, Skv, d, scale, *, ldq=None, ldk=None,
                  ldv=None, lddq=None, lddk=None, lddv=None, q_off=0, k_off=0, v_off=0, dq_off=0, dk_off=0, dv_off=0,
                  ws=None):
    """dq/dk/dv (bf16) of attention(); q/k/v and dq/dk/dv may be column slices (buffer + element offset)."""
    _chk(q, k, v, out, dout, lse, dq, dk, dv)
    need = attention_bwd_workspace_bytes(batch, heads, Sq)
    if ws is None or ws.numel() < need:
        ws = _workspace("attn_bwd", need, q.device, zero=False)
    check(lib().b200sd_attention_bwd(q.data_ptr() + q_off * 2, k.data_ptr() + k_off * 2, v.data_ptr() + v_off * 2,
                                     _p(out), _p(dout), _p(lse), dq.data_ptr() + dq_off * 2, dk.data_ptr() + dk_off * 2,
                                     dv.data_ptr() + dv_off * 2, batch, heads, Sq, Skv, d, ldq or q.shape[-1],
                                     ldk or k.shape[-1], ldv or v.shape[-1], out.shape[-1], dout.shape[-1],
                                     lddq or dq.shape[-1], lddk or dk.shape[-1], lddv or dv.shape[-1], float(scale),
                                     _p(ws), ws.numel(), _stream()), "attention_bwd")


def grad_prep(g, out_bf16=None, colsum=None, rows_per_image=0, ldcs=0, rows=None, N=None, ld=None):
    """optional bf16 copy of gradient g [rows, N] + column sums accumulated into colsum (bias gradient).
    rows / N / ld describe a column window of a wider row-major buffer when g is a flat slice."""
    _chk(g, out_bf16, colsum)
    if N is None:
        N = g.shape[-1]
    if rows is None:
        rows = g.numel() // N
    check(lib().b200sd_grad_prep(_p(g), _dt(g), _p(out_bf16), _p(colsum), rows, N, ld or N, rows_per_image, ldcs,
                                 _stream()), "grad_prep")
    return out_bf16


def cast_flat(src_f32, dst_bf16):
    _chk(src_f32, dst_bf16)
    check(lib().b200sd_cast_flat(_p(src_f32), _p(dst_bf16), src_f32.numel(), _stream()), "cast_flat")
    return dst_bf16


def adamw_step(param, grad, exp_avg, exp_avg_sq, weights_bf16, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0,
               zero_grad=False):
    _chk(param, grad, exp_avg, exp_avg_sq, weights_bf16)
    check(lib().b200sd_adamw_step(_p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), _p(weights_bf16), param.numel(),
                                  float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step),
                                  float(grad_scale), int(zero_grad), _stream()), "adamw_step")


def adamw8bit_step(param, grad, state1, state2, absmax1, absmax2, qmap1, qmap2, chunk_mode, small_exp_avg, small_exp_avg_sq,
                   weights_bf16, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0, zero_grad=False):
    """bnb.optim.AdamW8bit semantics over a flat buffer (include/b200sd.h: b200sd_adamw8bit_step)"""
    _chk(param, grad, state1, state2, absmax1, absmax2, qmap1, qmap2, chunk_mode, small_exp_avg, small_exp_avg_sq, weights_bf16)
    check(lib().b200sd_adamw8bit_step(_p(param), _p(grad), _p(state1), _p(state2), _p(absmax1), _p(absmax2), _p(qmap1), _p(qmap2),
                                      _p(chunk_mode), _p(small_exp_avg), _p(small_exp_avg_sq), _p(weights_bf16), param.numel(),
                                      float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step),
                                      float(grad_scale), int(zero_grad), _stream()), "adamw8bit_step")


def groupnorm_silu_bwd(x0, x1, gamma, beta, dy, out0, out1, batch, hw, *, add_src=None, acc0=False, acc1=False,
                       dgamma=None, dbeta=None, groups=32, eps=1e-5, silu=True, mean_rstd=None):
    _chk(x0, x1, gamma, beta, dy, out0, out1, add_src, dgamma, dbeta, mean_rstd)
    ws = _workspace("gn_bwd", lib().b200sd_groupnorm_bwd_workspace_floats(batch) * 4, x0.device, zero=True)
    C0 = x0.shape[-1]
    C1 = x1.shape[-1] if x1 is not None else 0
    check(lib().b200sd_groupnorm_silu_bwd(_p(x0), _p(x1), C0, C1, _dt(x0), _p(gamma), _p(beta), _p(dy), _p(add_src),
                                          _p(out0), _p(out1), _dt(out0), int(acc0), int(acc1), _p(dgamma), _p(dbeta),
                                          _p(mean_rstd), _p(ws), batch, hw, groups, float(eps), int(silu), _stream()),
          "groupnorm_silu_bwd")


def layernorm_bwd(x, gamma, dy, dres, dgamma=None, dbeta=None, eps=1e-5):
    _chk(x, gamma, dy, dres, dgamma, dbeta)
    Cc = x.shape[-1]
    check(lib().b200sd_layernorm_bwd(_p(x), _dt(x), _p(gamma), _p(dy), _p(dres), _p(dgamma), _p(dbeta), x.numel() // Cc,
                                     Cc, float(eps), _stream()), "layernorm_bwd")


def geglu_fwd(u, out):
    _chk(u, out)
    check(lib().b200sd_geglu_fwd(_p(u), _p(out), u.numel() // u.shape[-1], u.shape[-1] // 2, _stream()), "geglu_fwd")
    return out


def geglu_bwd(u, dff, du):
    _chk(u, dff, du)
    check(lib().b200sd_geglu_bwd(_p(u), _p(dff), _p(du), u.numel() // u.shape[-1], u.shape[-1] // 2, _stream()),
          "geglu_bwd")
    return du


def upsample2x_bwd(dy, dx, batch, H, W, accumulate=False):
    _chk(dy, dx)
    check(lib().b200sd_upsample2x_bwd(_p(dy), _p(dx), batch, H, W, dx.shape[-1], int(accumulate), _stream()),
          "upsample2x_bwd")


def col2im_s2(dcol, dx, batch, H, W, accumulate=False):
    _chk(dcol, dx)
    check(lib().b200sd_col2im_s2(_p(dcol), _p(dx), batch, H, W, dx.shape[-1], int(accumulate), _stream()), "col2im_s2")


def conv_out_bwd(dout_nchw, x_nhwc, w_packed, dx_nhwc, dw=None, dbias=None):
    _chk(dout_nchw, x_nhwc, w_packed, dx_nhwc, dw, dbias)
    B, Cout, H, W = dout_nchw.shape
    check(lib().b200sd_conv_out_bwd(_p(dout_nchw), _p(x_nhwc), _p(w_packed), _p(dx_nhwc), _p(dw), _p(dbias), B,
                                    dx_nhwc.shape[-1], Cout, H, W, _stream()), "conv_out_bwd")


def conv_in_wgrad(dy_nhwc, x_nchw, dw):
    _chk(dy_nhwc, x_nchw, dw)
    B, Cin, H, W = x_nchw.shape
    check(lib().b200sd_conv_in_wgrad(_p(dy_nhwc), _dt(dy_nhwc), _p(x_nchw), _p(dw), B, Cin, dy_nhwc.shape[-1], H, W,
                                     _stream()), "conv_in_wgrad")


def cast_act(x, out_bf16, silu=False):
    _chk(x, out_bf16)
    check(lib().b200sd_cast_act(_p(x), _p(out_bf16), x.numel(), int(silu), _stream()), "cast_act")
    return out_bf16


def silu_bwd_mul(pre, grad):
    _chk(pre, grad)
    check(lib().b200sd_silu_bwd_mul(_p(pre), _p(grad), grad.numel(), _stream()), "silu_bwd_mul")
    return grad


# ---------------------------------------------------------------------------------------------
# fp32-accuracy path: operands travel as (hi, lo) bf16 pairs, products are 3-term (see include/b200sd.h)
# ---------------------------------------------------------------------------------------------
def split_hi_lo(x, hi, lo):
    _chk(x, hi, lo)
    check(lib().b200sd_split_hi_lo(_p(x), _p(hi), _p(lo), x.numel(), _stream()), "split_hi_lo")


def groupnorm_silu_split(x0, x1, gamma, beta, out, out_lo, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None, raw_lo=None):
    _chk(x0, x1, gamma, beta, out, out_lo, raw_out, raw_lo)
    if x1 is not None and x1.dtype != x0.dtype:
        raise B200SDError("groupnorm: both sources must have the same dtype")
    ws = _workspace(("gn", _stream()), lib().b200sd_groupnorm_workspace_floats(batch) * 4, x0.device)
    C0 = x0.shape[-1]
    C1 = x1.shape[-1] if x1 is not None else 0
    check(lib().b200sd_groupnorm_silu_split(_p(x0), _p(x1), C0, C1, _p(gamma), _p(beta), _p(out), _p(out_lo), _p(raw_out),
                                            _p(raw_lo), _p(ws), None, batch, hw, groups, float(eps), int(silu), _dt(x0),
                                            _stream()), "groupnorm_silu_split")


def layernorm_split(x, gamma, beta, out, out_lo, eps=1e-5):
    _chk(x, gamma, beta, out, out_lo)
    Cc = x.shape[-1]
    check(lib().b200sd_layernorm_split(_p(x), _p(gamma), _p(beta), _p(out), _p(out_lo), x.numel() // Cc, Cc, float(eps), _dt(x),
                                       _stream()), "layernorm_split")


def geglu_f32(u, hi, lo):
    _chk(u, hi, lo)
    check(lib().b200sd_geglu_f32(_p(u), _p(hi), _p(lo), u.numel() // u.shape[-1], u.shape[-1] // 2, _stream()), "geglu_f32")


def attention_f32(q, k, v, out, batch, heads, Sq, Skv, d, scale, ldq=None, ldk=None, ldv=None, ldo=None, q_off=0, k_off=0, v_off=0):
    _chk(q, k, v, out)
    check(lib().b200sd_attention_f32(q.data_ptr() + q_off * 4, k.data_ptr() + k_off * 4, v.data_ptr() + v_off * 4, _p(out), batch,
                                     heads, Sq, Skv, d, ldq or q.shape[-1], ldk or k.shape[-1], ldv or v.shape[-1],
                                     ldo or out.shape[-1], float(scale), _stream()), "attention_f32")


def small_linear_f32(x, w, bias, silu_in=False, silu_out=False, out=None):
    _chk(x, w, bias, out)
    B, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(B, N, dtype=torch.float32, device=x.device)
    check(lib().b200sd_small_linear_f32(_p(x), _p(w), _p(bias), _p(out), B, N, K, int(silu_in), int(silu_out), _stream()),
          "small_linear_f32")
    return out


# ---------------------------------------------------------------------------------------------
# CLIP text encoder (SURVEY.md 8f N3)
# ---------------------------------------------------------------------------------------------
def clip_embed(ids, tok, pos, out):
    _chk(ids, tok, pos, out)
    B, S = ids.shape
    check(lib().b200sd_clip_embed(_p(ids), _p(tok), _p(pos), _p(out), B, S, tok.shape[1], tok.shape[0], _stream()), "clip_embed")
    return out


def clip_embed_bwd(ids, dx, dtok, dpos):
    _chk(ids, dx, dtok, dpos)
    B, S = ids.shape
    check(lib().b200sd_clip_embed_bwd(_p(ids), _p(dx), _p(dtok), _p(dpos), B, S, dtok.shape[1], dtok.shape[0], _stream()),
          "clip_embed_bwd")


def quick_gelu_fwd(u, out):
    _chk(u, out)
    check(lib().b200sd_quick_gelu_fwd(_p(u), _p(out), u.numel(), _stream()), "quick_gelu_fwd")
    return out


def quick_gelu_bwd(u, dg, du):
    _chk(u, dg, du)
    check(lib().b200sd_quick_gelu_bwd(_p(u), _p(dg), _p(du), u.numel(), _stream()), "quick_gelu_bwd")
    return du


def layernorm_f32out(x, gamma, beta, out, eps=1e-5):
    _chk(x, gamma, beta, out)
    if x.dtype != torch.float32 or out.dtype != torch.float32:
        raise B200SDError("layernorm_f32out: fp32 in, fp32 out")
    Cc = x.shape[-1]
    check(lib().b200sd_layernorm_f32out(_p(x), _p(gamma), _p(beta), _p(out), x.numel() // Cc, Cc, float(eps), _stream()),
          "layernorm_f32out")
    return out


def causal_attention(qkv, out, batch, heads, S, d, scale):
    """qkv bf16 [batch*S, 3*heads*d] = [q | k | v]; out bf16 [batch*S, heads*d]"""
    _chk(qkv, out)
    Cc = heads * d
    check(lib().b200sd_causal_attention(_p(qkv), _p(out), batch, heads, S, d, qkv.shape[-1], out.shape[-1], 0, Cc, 2 * Cc,
                                        float(scale), _stream()), "causal_attention")
    return out


def causal_attention_bwd(qkv, dout, dqkv, batch, heads, S, d, scale):
    _chk(qkv, dout, dqkv)
    Cc = heads * d
    check(lib().b200sd_causal_attention_bwd(_p(qkv), _p(dout), _p(dqkv), batch, heads, S, d, qkv.shape[-1], dout.shape[-1],
                                            dqkv.shape[-1], 0, Cc, 2 * Cc, float(scale), _stream()), "causal_attention_bwd")
    return dqkv


# ---------------------------------------------------------------------------------------------
# AutoencoderKL (SURVEY.md 8f N1)
# ---------------------------------------------------------------------------------------------
def softmax_rows(x, out, scale=1.0):
    """x fp32 [rows, L] -> out bf16 [rows, L] = softmax(scale * x) along the last dim"""
    _chk(x, out)
    rows, L = x.shape
    check(lib().b200sd_softmax_rows(_p(x), _p(out), rows, L, x.shape[-1], out.shape[-1], float(scale), _stream()), "softmax_rows")
    return out


def conv1x1_small(x_nchw, w, bias, out_nchw):
    _chk(x_nchw, w, bias, out_nchw)
    B, Cin, H, W = x_nchw.shape
    check(lib().b200sd_conv1x1_small(_p(x_nchw), _p(w), _p(bias), _p(out_nchw), B, Cin, w.shape[0], H * W, _stream()), "conv1x1_small")
    return out_nchw


def gaussian_sample(moments, noise, out, out_scale=1.0):
    _chk(moments, noise, out)
    B, C2, H, W = moments.shape
    check(lib().b200sd_gaussian_sample(_p(moments), _p(noise), _p(out), B, C2 // 2, H * W, float(out_scale), _stream()), "gaussian_sample")
    return out
