"""fp32-accuracy launch plan of one UNet forward (BASELINE north_star: "the fp32 path within 1e-4").

Same structure as engine.py (static plan of C-ABI calls over pre-allocated NHWC buffers, CUDA-graph replay), but
every tensor between kernels is fp32 and every contraction is evaluated to ~fp32 accuracy ON THE bf16 TENSOR CORES:
an fp32 operand x travels as the pair (hi, lo) = (bf16(x), bf16(x - hi)) and

    A B^T  ~=  A_hi B_hi^T + A_lo B_hi^T + A_hi B_lo^T          (the dropped lo*lo term is ~2^-18 relative)

is two launches of the SAME tcgen05 GEMM / implicit-GEMM conv kernel with fp32 accumulation:
    (1) [A_hi | A_lo] x [B_hi | B_hi]^T   -- the kernel's two-source K concat (per tap for conv3x3), + bias / time
                                              embedding / residual in the epilogue, fp32 out
    (2)  A_hi x B_lo^T                     -- accumulated in place through the fp32 residual input.
GroupNorm / LayerNorm emit (hi, lo) directly, GEGLU runs on the fp32 pre-activation, attention is an fp32 CUDA-core
flash kernel, the time-embedding linears use fp32 weights.  ~3x the tensor-core work of the bf16 plan plus the fp32
attention: an accuracy path, selected with `unet.set_precision("fp32")`.
"""
from __future__ import annotations

import torch

from . import ops
from .engine import Engine

F32, BF16 = torch.float32, torch.bfloat16


def _split(w2d: torch.Tensor):
    w2d = w2d.detach().float().contiguous()
    hi = w2d.to(BF16)
    lo = (w2d - hi.float()).to(BF16)
    return hi, lo


def _pack_conv(w):      # (Cout, Cin, 3, 3) -> W1 [Cout][9][2Cin] = per tap [hi | hi], W2 [Cout][9][Cin] = lo
    co, ci = w.shape[0], w.shape[1]
    hi, lo = _split(w.detach().permute(0, 2, 3, 1).reshape(co, 9 * ci))
    hi3 = hi.view(co, 9, ci)
    return torch.cat([hi3, hi3], dim=2).reshape(co, 18 * ci).contiguous(), lo.contiguous()


def _pack_lin(w):       # (out, in[,1,1]) -> W1 [out][2 in] = [hi | hi], W2 [out][in] = lo
    hi, lo = _split(w.detach().reshape(w.shape[0], -1))
    return torch.cat([hi, hi], dim=1).contiguous(), lo.contiguous()


class EngineF32(Engine):
    """Engine's inputs, context cache and execution over the fp32-accuracy plan built below."""

    def _buf(self, rows, cols, dtype=F32):
        return torch.empty(rows, cols, dtype=dtype, device=self.device)

    def _pair(self, rows, cols):
        return self._buf(rows, cols, BF16), self._buf(rows, cols, BF16)

    def _gemm2(self, plan, a_hi, a_lo, w12, out, *, bias=None, residual=None, conv=None, rowbias_ptr=None):
        """out (fp32) = A W^T (+bias +rowbias +residual) to ~fp32 accuracy: two launches of the bf16 tensor-core GEMM"""
        w1, w2 = w12
        self.gemm(plan, a_hi, w1, out, a1=a_lo, bias=bias, residual=residual, conv=conv, rowbias_ptr=rowbias_ptr)
        self.gemm(plan, a_hi, w2, out, residual=out, conv=conv)

    def _build(self):
        m, N, dev = self.model, self.N, self.device
        cfg = m.config
        boc = cfg.block_out_channels
        P = self.plan
        eps = cfg.norm_eps
        heads = self.heads
        f32p = lambda t: t.detach().float().contiguous()

        self.in_sample = torch.zeros(N, cfg.in_channels, self.H, self.W, dtype=F32, device=dev)
        self.in_t = torch.zeros(N, dtype=F32, device=dev)
        self.in_ctx = torch.zeros(N * self.S, self.ctx_dim, dtype=F32, device=dev)
        self.out = torch.zeros(N, cfg.out_channels, self.H, self.W, dtype=F32, device=dev)
        ctx_hi, ctx_lo = self._pair(N * self.S, self.ctx_dim)
        self.ctx_plan.append(lambda: ops.split_hi_lo(self.in_ctx, ctx_hi, ctx_lo))

        # ---- time embedding: everything fp32 ----
        te = m.time_embedding
        resnets = list(m._iter_resnets())
        tp_w = torch.cat([f32p(r.time_emb_proj.weight) for _, r in resnets], 0)
        tp_b = torch.cat([f32p(r.time_emb_proj.bias) for _, r in resnets], 0)
        tp_off, n_tp = m._tproj_offsets()
        temb_dim = boc[0] * 4
        t_sin = self._buf(N, boc[0])
        t_h = self._buf(N, temb_dim)
        t_emb = self._buf(N, temb_dim)
        self.tproj = self._buf(N, n_tp)
        w1, b1, w2, b2 = f32p(te.linear_1.weight), f32p(te.linear_1.bias), f32p(te.linear_2.weight), f32p(te.linear_2.bias)
        P.append(lambda: ops.timestep_embedding(self.in_t, boc[0], out=t_sin))
        P.append(lambda: ops.small_linear_f32(t_sin, w1, b1, silu_out=True, out=t_h))
        P.append(lambda: ops.small_linear_f32(t_h, w2, b2, out=t_emb))
        P.append(lambda: ops.small_linear_f32(t_emb, tp_w, tp_b, silu_in=True, out=self.tproj))

        def resnet(prefix, r, x, skip, h, w):
            M, hw = N * h * w, h * w
            cin, cout = r.cin, r.cout
            has_sc = hasattr(r, "conv_shortcut")
            g1, be1, g2, be2 = f32p(r.norm1.weight), f32p(r.norm1.bias), f32p(r.norm2.weight), f32p(r.norm2.bias)
            t1h, t1l = self._pair(M, cin)
            rawh, rawl = self._pair(M, cin) if has_sc else (None, None)
            P.append(lambda: ops.groupnorm_silu_split(x, skip, g1, be1, t1h, t1l, N, hw, 32, eps, True, raw_out=rawh, raw_lo=rawl))
            hbuf = self._buf(M, cout)
            rb = (self.tproj.data_ptr() + tp_off[prefix] * 4, n_tp, hw)
            self._gemm2(P, t1h, t1l, _pack_conv(r.conv1.weight), hbuf, bias=f32p(r.conv1.bias), conv=(N, h, w), rowbias_ptr=rb)
            t2h, t2l = self._pair(M, cout)
            P.append(lambda: ops.groupnorm_silu_split(hbuf, None, g2, be2, t2h, t2l, N, hw, 32, eps, True))
            if has_sc:
                sc = self._buf(M, cout)
                self._gemm2(P, rawh, rawl, _pack_lin(r.conv_shortcut.weight), sc, bias=f32p(r.conv_shortcut.bias))
            else:
                sc = x
            y = self._buf(M, cout)
            self._gemm2(P, t2h, t2l, _pack_conv(r.conv2.weight), y, bias=f32p(r.conv2.bias), residual=sc, conv=(N, h, w))
            return y

        def xformer(prefix, a, x, h, w):
            blk = a.transformer_blocks[0]
            Cc = a.ch
            M, hw = N * h * w, h * w
            d = Cc // heads
            scale = d ** -0.5
            S = self.S
            a1m, a2m, ff = blk.attn1, blk.attn2, blk.ff
            kv = self._buf(N * S, 2 * Cc)
            self._gemm2(self.ctx_plan, ctx_hi, ctx_lo, _pack_lin(torch.cat([a2m.to_k.weight, a2m.to_v.weight], 0)), kv)
            th, tl = self._pair(M, Cc)
            gn_g, gn_b = f32p(a.norm.weight), f32p(a.norm.bias)
            P.append(lambda: ops.groupnorm_silu_split(x, None, gn_g, gn_b, th, tl, N, hw, 32, 1e-6, False))
            hs0 = self._buf(M, Cc)
            self._gemm2(P, th, tl, _pack_lin(a.proj_in.weight), hs0, bias=f32p(a.proj_in.bias))
            nh, nl = self._pair(M, Cc)
            ah, al = self._pair(M, Cc)
            at = self._buf(M, Cc)
            ln = [(f32p(n.weight), f32p(n.bias)) for n in (blk.norm1, blk.norm2, blk.norm3)]
            # self attention
            P.append(lambda: ops.layernorm_split(hs0, ln[0][0], ln[0][1], nh, nl))
            qkv = self._buf(M, 3 * Cc)
            self._gemm2(P, nh, nl, _pack_lin(torch.cat([a1m.to_q.weight, a1m.to_k.weight, a1m.to_v.weight], 0)), qkv)
            P.append(lambda: ops.attention_f32(qkv, qkv, qkv, at, N, heads, hw, hw, d, scale, ldq=3 * Cc, ldk=3 * Cc, ldv=3 * Cc, ldo=Cc,
                                               k_off=Cc, v_off=2 * Cc))
            P.append(lambda: ops.split_hi_lo(at, ah, al))
            hs1 = self._buf(M, Cc)
            self._gemm2(P, ah, al, _pack_lin(a1m.to_out[0].weight), hs1, bias=f32p(a1m.to_out[0].bias), residual=hs0)
            # cross attention
            P.append(lambda: ops.layernorm_split(hs1, ln[1][0], ln[1][1], nh, nl))
            q2 = self._buf(M, Cc)
            self._gemm2(P, nh, nl, _pack_lin(a2m.to_q.weight), q2)
            P.append(lambda: ops.attention_f32(q2, kv, kv, at, N, heads, hw, S, d, scale, ldq=Cc, ldk=2 * Cc, ldv=2 * Cc, ldo=Cc, v_off=Cc))
            P.append(lambda: ops.split_hi_lo(at, ah, al))
            hs2 = self._buf(M, Cc)
            self._gemm2(P, ah, al, _pack_lin(a2m.to_out[0].weight), hs2, bias=f32p(a2m.to_out[0].bias), residual=hs1)
            # GEGLU feed-forward on the fp32 pre-activation
            P.append(lambda: ops.layernorm_split(hs2, ln[2][0], ln[2][1], nh, nl))
            u = self._buf(M, 8 * Cc)
            self._gemm2(P, nh, nl, _pack_lin(ff.net[0].proj.weight), u, bias=f32p(ff.net[0].proj.bias))
            fh, fl = self._pair(M, 4 * Cc)
            P.append(lambda: ops.geglu_f32(u, fh, fl))
            hs3 = self._buf(M, Cc)
            self._gemm2(P, fh, fl, _pack_lin(ff.net[2].weight), hs3, bias=f32p(ff.net[2].bias), residual=hs2)
            P.append(lambda: ops.split_hi_lo(hs3, ah, al))
            y = self._buf(M, Cc)
            self._gemm2(P, ah, al, _pack_lin(a.proj_out.weight), y, bias=f32p(a.proj_out.bias), residual=x)
            return y

        def resample(x, h, w, down):
            Cc = x.shape[1]
            xh, xl = self._pair(x.shape[0], Cc)
            P.append(lambda: ops.split_hi_lo(x, xh, xl))
            if down:
                rows, cols = N * (h // 2) * (w // 2), 9 * Cc
                oh, ol = self._pair(rows, cols)
                P.append(lambda: ops.im2col_s2(xh, oh, N, h, w))
                P.append(lambda: ops.im2col_s2(xl, ol, N, h, w))
            else:
                oh, ol = self._pair(N * 4 * h * w, Cc)
                P.append(lambda: ops.upsample2x(xh, oh, N, h, w))
                P.append(lambda: ops.upsample2x(xl, ol, N, h, w))
            return oh, ol

        def downsample(_prefix, s, x, h, w):
            ds = s.conv
            ch, cl = resample(x, h, w, True)
            y = self._buf(N * (h // 2) * (w // 2), x.shape[1])
            wp = ds.weight.detach().permute(0, 2, 3, 1).reshape(ds.weight.shape[0], -1)      # [Cout][9*Cin] matches im2col order
            self._gemm2(P, ch, cl, _pack_lin(wp), y, bias=f32p(ds.bias))
            return y

        def upsample(_prefix, s, x, h, w):
            us = s.conv
            uh, ul = resample(x, h, w, False)
            y = self._buf(N * 4 * h * w, x.shape[1])
            self._gemm2(P, uh, ul, _pack_conv(us.weight), y, bias=f32p(us.bias), conv=(N, 2 * h, 2 * w))
            return y

        # ---- forward graph ----
        h, w = self.H, self.W
        x = self._buf(N * h * w, boc[0])
        ci_w, ci_b = f32p(m.conv_in.weight.detach().permute(0, 2, 3, 1).reshape(boc[0], -1)), f32p(m.conv_in.bias)
        P.append(lambda x=x: ops.conv_in(self.in_sample, ci_w, ci_b, x))
        x, h, w = m._walk(x, h, w, resnet=resnet, xformer=xformer, downsample=downsample, upsample=upsample, release=lambda t: None)
        # ---- out: GroupNorm+SiLU -> (hi, lo); the 4-channel conv is linear, so conv(hi) + conv(lo) with fp32 weights ----
        th, tl = self._pair(N * h * w, boc[0])
        go, bo = f32p(m.conv_norm_out.weight), f32p(m.conv_norm_out.bias)
        x_last = x
        P.append(lambda: ops.groupnorm_silu_split(x_last, None, go, bo, th, tl, N, h * w, 32, eps, True))
        co_w = f32p(m.conv_out.weight.detach().permute(0, 2, 3, 1).reshape(cfg.out_channels, -1))
        co_b, zero_b = f32p(m.conv_out.bias), torch.zeros(cfg.out_channels, dtype=F32, device=dev)
        out_lo = torch.zeros_like(self.out)
        P.append(lambda: ops.conv_out(th, co_w, co_b, self.out))
        P.append(lambda: ops.conv_out(tl, co_w, zero_b, out_lo))
        P.append(lambda: self.out.add_(out_lo))
