"""Training engine: forward-with-saved-activations and backward launch plans of the UNet (SURVEY.md row A9:
`accelerator.backward(loss)` through `unet(noisy_latents, timesteps, encoder_hidden_states)`,
finetune_sd.py:480-494), for a fixed (batch, H, W, ctx_len) geometry.

Like engine.py every plan entry is one C-ABI call into libb200sd.so over pre-allocated NHWC buffers;
nothing is allocated at run time.  What differs from the inference plan:
  * every tensor the backward needs is kept (no buffer recycling across the forward), attention also
    writes its log-sum-exp, GEGLU keeps its pre-activation, the time MLP keeps pre-SiLU values;
  * weights live in ONE flat bf16 buffer in kernel layout (refreshed from the fp32 parameters with a
    multi-tensor copy when they change) and ALL parameter gradients are accumulated by the kernels into
    ONE flat fp32 buffer in the same order -- the unit the data-parallel allreduce and a fused optimizer
    work on.  `param.grad` tensors are views of that buffer (permuted for 3x3 conv weights, whose
    kernel layout is [Cout][ky][kx][Cin]).

Backward data flow per block (each arrow = one kernel; dW = wgrad GEMM, dX = dgrad GEMM):
  resnet : dy -prep-> dy16 (+dbias) ; dW2(t2, dy16) ; dX2 -> dt2 -GN'-> dh16 (+dtemb) ; dW1(t1, dh16) ; dX1 -> dt1
           [shortcut: dWsc(raw, dy16) ; dXsc -> dsc]  -GN'(+ dsc | dy)-> dx, dskip
  xformer: dy -prep-> dy16 ; dWout ; dXout -> dhs ; per sub-layer: prep(dhs) ; dW, dX of the output linear ;
           (attention' | GEGLU') ; dW, dX of the input linears ; LN' accumulates into dhs ;
           finally dWin ; dXin -> dt -GN'(+dy)-> dx
"""
from __future__ import annotations

import torch

from . import ops
from ._lib import B200SDError
from .plan import Builder, Plan, Pool

F32, BF16 = torch.float32, torch.bfloat16
_ALIGN = 64  # elements: every region starts 128-byte aligned in the bf16 buffer (TMA needs 16)


class _Reg:
    """One parameter inside the flat buffers."""
    __slots__ = ("param", "kind", "off", "numel", "shape2d", "g", "gview", "wb", "wf", "pview", "rehomed", "src")


class FlatParams:
    """Flat kernel-layout state of a UNet2DConditionModel, all in ONE order (execution order of the forward, the
    time-embedding parameters first -- their gradients complete last in the backward):
       master fp32  the parameters themselves: every `nn.Parameter.data` is re-homed to a view of this buffer
                    ([Cout][ky][kx][Cin] for 3x3 convs, i.e. a permuted view of the diffusers OIHW shape; fused q|k|v,
                    k|v and the 22 time_emb_proj heads are adjacent so one GEMM reads them as one matrix)
       wb     bf16  tensor-core copy of master (one cast kernel, or written by the fused AdamW step)
       grad   fp32  every parameter's gradient (accumulated by the backward kernels)
    state_dict() / load_state_dict() / torch optimizers keep working on the re-homed parameters."""

    def __init__(self, model, device, lazy=False, allow_half_trainable=False):
        self.model, self.device = model, device
        self.regs = {}        # id(param) -> _Reg
        self.order = []
        off = 0

        def add(p, kind):
            nonlocal off
            if p.dtype != F32 and p.requires_grad and not allow_half_trainable:
                raise B200SDError("training needs fp32 master parameters (the kernels compute in bf16 on their own copy)")
            r = _Reg()
            # a FROZEN fp16 / bf16 parameter (finetune_sd.py:393: unet.to(device, dtype=torch.float16) while the text encoder
            # trains) keeps its own storage; the flat fp32 master holds an upcast copy for the kernels
            r.rehomed = p.dtype == F32
            r.param, r.kind, r.numel = p, kind, p.numel()
            r.off = off
            off += (p.numel() + _ALIGN - 1) // _ALIGN * _ALIGN
            self.regs[id(p)] = r
            self.order.append(r)
            return r

        def add_adjacent(ps, kind):
            """regions packed back to back (no padding in between): requires numel % _ALIGN == 0"""
            for p in ps:
                if p.numel() % _ALIGN:
                    raise B200SDError("fused weight regions must be multiples of 64 elements")
                add(p, kind)

        m = model
        self._layout(model, add, add_adjacent)
        missing = [n for n, p in m.named_parameters() if id(p) not in self.regs]
        if missing:
            raise B200SDError(f"FlatParams: parameters not laid out: {missing[:4]}...")
        self.total = off
        self.master = torch.zeros(off, dtype=F32, device=device)
        self.grad = self.wb = None           # allocated by materialize() at the first training forward
        for r in self.order:
            p = r.param
            mst = self.master[r.off:r.off + r.numel]
            r.wb = r.wf = r.g = r.gview = None
            if r.kind in ("conv3", "conv_f32"):
                co, ci, kh, kw = p.shape
                r.shape2d = (co, kh * kw * ci)
                r.pview = mst.view(co, kh, kw, ci).permute(0, 3, 1, 2)
                if r.kind == "conv_f32":
                    r.wf = mst.view(r.shape2d)       # the CUDA-core end convs read the fp32 master directly
            elif r.kind == "lin":
                r.shape2d = (p.shape[0], p.numel() // p.shape[0])
                r.pview = mst.view(p.shape)
            else:
                r.shape2d = (p.numel(),)
                r.pview = mst.view(p.shape)
        # re-home the parameters into the flat master buffer (Parameter identity is preserved)
        with torch.no_grad():
            for r in self.order:
                r.pview.copy_(r.param.data)
                if r.rehomed:
                    r.param.data = r.pview
                r.src = (r.param.data.data_ptr(), r.param.dtype)
        self._versions = None
        if not lazy:
            self.materialize()

    def _layout(self, m, add, add_adjacent):
        """Register every parameter of the model, in the order the forward uses them (subclasses: other model families)."""
        def add_resnet(r):
            add(r.norm1.weight, "vec"); add(r.norm1.bias, "vec")
            add(r.conv1.weight, "conv3"); add(r.conv1.bias, "vec")
            add(r.norm2.weight, "vec"); add(r.norm2.bias, "vec")
            add(r.conv2.weight, "conv3"); add(r.conv2.bias, "vec")
            if hasattr(r, "conv_shortcut"):
                add(r.conv_shortcut.weight, "lin"); add(r.conv_shortcut.bias, "vec")

        def add_xformer(a):
            blk = a.transformer_blocks[0]
            add(a.norm.weight, "vec"); add(a.norm.bias, "vec")
            add(a.proj_in.weight, "lin"); add(a.proj_in.bias, "vec")
            for n in (blk.norm1, blk.norm2, blk.norm3):
                add(n.weight, "vec"); add(n.bias, "vec")
            add_adjacent([blk.attn1.to_q.weight, blk.attn1.to_k.weight, blk.attn1.to_v.weight], "lin")
            add(blk.attn1.to_out[0].weight, "lin"); add(blk.attn1.to_out[0].bias, "vec")
            add(blk.attn2.to_q.weight, "lin")
            add_adjacent([blk.attn2.to_k.weight, blk.attn2.to_v.weight], "lin")
            add(blk.attn2.to_out[0].weight, "lin"); add(blk.attn2.to_out[0].bias, "vec")
            add(blk.ff.net[0].proj.weight, "lin"); add(blk.ff.net[0].proj.bias, "vec")
            add(blk.ff.net[2].weight, "lin"); add(blk.ff.net[2].bias, "vec")
            add(a.proj_out.weight, "lin"); add(a.proj_out.bias, "vec")

        def add_sampler(s):
            add(s.conv.weight, "conv3"); add(s.conv.bias, "vec")

        te = m.time_embedding
        add(te.linear_1.weight, "lin"); add(te.linear_1.bias, "vec")
        add(te.linear_2.weight, "lin"); add(te.linear_2.bias, "vec")
        resnets = list(m._iter_resnets())
        add_adjacent([r.time_emb_proj.weight for _, r in resnets], "lin")
        add_adjacent([r.time_emb_proj.bias for _, r in resnets], "vec")
        add(m.conv_in.weight, "conv_f32"); add(m.conv_in.bias, "vec")
        for b in m.down_blocks:
            for j, r in enumerate(b.resnets):
                add_resnet(r)
                if hasattr(b, "attentions"):
                    add_xformer(b.attentions[j])
            if hasattr(b, "downsamplers"):
                add_sampler(b.downsamplers[0])
        add_resnet(m.mid_block.resnets[0]); add_xformer(m.mid_block.attentions[0]); add_resnet(m.mid_block.resnets[1])
        for b in m.up_blocks:
            for j, r in enumerate(b.resnets):
                add_resnet(r)
                if hasattr(b, "attentions"):
                    add_xformer(b.attentions[j])
            if hasattr(b, "upsamplers"):
                add_sampler(b.upsamplers[0])
        add(m.conv_norm_out.weight, "vec"); add(m.conv_norm_out.bias, "vec")
        add(m.conv_out.weight, "conv_f32"); add(m.conv_out.bias, "vec")


    def materialize(self):
        """Allocate the training-only state: the flat fp32 gradient buffer and the bf16 tensor-core copy of the weights.  (The
        master buffer alone is set up as soon as the model lands on the GPU -- unet.to(device) -- so that whoever wraps the model
        afterwards, e.g. DistributedDataParallel via accelerator.prepare (finetune_sd.py:363, 386), sees the parameters' FINAL
        strides: the 3x3 conv weights are permuted views of their kernel-layout storage.)"""
        if self.grad is not None:
            return self
        dev = self.master.device
        self.grad = torch.zeros(self.total, dtype=F32, device=dev)
        self.wb = torch.zeros(self.total, dtype=BF16, device=dev)
        for r in self.order:
            p = r.param
            sl = slice(r.off, r.off + r.numel)
            g, w = self.grad[sl], self.wb[sl]
            if r.kind in ("conv3", "conv_f32"):
                co, ci, kh, kw = p.shape
                r.g = g.view(r.shape2d)
                r.gview = g.view(co, kh, kw, ci).permute(0, 3, 1, 2)
                if r.kind == "conv3":
                    r.wb = w.view(r.shape2d)
            elif r.kind == "lin":
                r.g, r.gview, r.wb = g.view(r.shape2d), g.view(p.shape), w.view(r.shape2d)
            else:
                r.g, r.gview = g, g.view(p.shape)
        self._versions = None
        return self

    def reg(self, p) -> _Reg:
        return self.regs[id(p)]

    def span(self, ps, buf):
        """one view over the adjacent regions of `ps` in flat buffer `buf` ("wb" | "grad" | "master")"""
        r0 = self.reg(ps[0])
        n = sum(p.numel() for p in ps)
        flat = getattr(self, buf)[r0.off:r0.off + n]
        return flat.view(-1, r0.shape2d[-1]) if len(r0.shape2d) == 2 else flat

    @torch.no_grad()
    def refresh_weights(self, force=False):
        """fp32 master -> bf16 tensor-core copy (one cast kernel over the flat buffer), only when a parameter changed."""
        ver = sum(r.param._version for r in self.order)
        if not force and ver == self._versions:
            return False
        for r in self.order:
            if not r.rehomed:           # frozen fp16 / bf16 parameter: the master holds an upcast COPY
                r.pview.copy_(r.param.data)
        ops.cast_flat(self.master, self.wb)
        self._versions = ver
        return True

    def zero_grad(self):
        self.grad.zero_()

    def attach_grads(self):
        """param.grad = view of the flat gradient buffer (same strides as the re-homed parameter)."""
        for r in self.order:
            if r.param.requires_grad:
                r.param.grad = r.gview

    def owns(self, model) -> bool:
        """True while every parameter still lives in the flat master buffer (a .to() / load of new tensors breaks it)."""
        base = self.master.untyped_storage().data_ptr()
        return all((r.param.data.untyped_storage().data_ptr() == base) if r.rehomed
                   else (r.param.data.data_ptr(), r.param.dtype) == r.src for r in self.order[:4] + self.order[-4:])


class TrainEngine(Builder):
    def __init__(self, model, flat: FlatParams, N, H, W, S_ctx, device, train_weights=True, ctx_grad=False):
        super().__init__(device)
        self.model, self.flat = model, flat
        self.N, self.H, self.W, self.S = N, H, W, S_ctx
        self.train_weights, self.ctx_grad = train_weights, ctx_grad
        cfg = model.config
        self.heads, self.ctx_dim = cfg.attention_head_dim, cfg.cross_attention_dim
        self.fwd, self.bwd = Plan(), Plan()
        self.ready_marks = []   # (number of backward entries executed, offset): flat.grad[offset:] is final
        self.saved_bytes = 0
        self._gi = {}      # id(activation) -> [grad buffer, initialised?]
        self.pool = Pool(device)
        with torch.cuda.device(device):
            self._build()

    # -- helpers ----------------------------------------------------------------------------------
    def _new(self, rows, cols, dtype=BF16):
        self.saved_bytes += rows * cols * (2 if dtype == BF16 else 4)
        return torch.empty(rows, cols, dtype=dtype, device=self.device)

    def _grad_of(self, t):
        """(grad buffer of residual-stream activation t, accumulate?) -- first writer overwrites, later ones add"""
        e = self._gi.get(id(t))
        if e is None:
            e = self._gi[id(t)] = [torch.empty_like(t, dtype=F32), False]
            self._keep.append(t)
        acc = e[1]
        e[1] = True
        return e[0], acc

    def _grad_ready(self, t):
        e = self._gi.get(id(t))
        if e is None or not e[1]:
            raise B200SDError("backward plan: gradient consumed before it was produced")
        return e[0]

    def G(self, p):
        """fp32 gradient region (kernel layout) of parameter p, or None when weights are frozen"""
        return self.flat.reg(p).g if self.train_weights else None

    def Wb(self, p):
        return self.flat.reg(p).wb

    def P(self, p):
        """fp32 view of parameter p in the flat master buffer -- what the kernels read for biases / norm affines.  (For a re-homed
        fp32 parameter this IS p.data; a frozen fp16 / bf16 parameter keeps its own storage and the master holds the upcast copy.)"""
        r = self.flat.reg(p)
        return r.pview if r.pview.is_contiguous() else r.param.data

    def _prep(self, g, want_bf16=True, bias_param=None, **kw):
        """bwd: bf16 copy of fp32 gradient g (+ bias gradient)"""
        out = self.pool.get(g.shape[0], g.shape[1]) if want_bf16 and g.dtype == F32 else None
        cs = self.G(bias_param) if bias_param is not None else None
        if out is not None or cs is not None:
            self.bwd.append(lambda: ops.grad_prep(g, out, cs, **kw))
        return out if out is not None else g

    # -- build ------------------------------------------------------------------------------------
    def _build(self):
        m, N, dev, flat = self.model, self.N, self.device, self.flat
        cfg = m.config
        boc = cfg.block_out_channels
        Fp, Bp = self.fwd, self.bwd
        f32 = dict(dtype=F32, device=dev)
        eps = cfg.norm_eps
        heads = self.heads
        tw = self.train_weights

        self.in_sample = torch.zeros(N, cfg.in_channels, self.H, self.W, **f32)
        self.in_t = torch.zeros(N, **f32)
        self.in_ctx = torch.zeros(N * self.S, self.ctx_dim, dtype=BF16, device=dev)
        self.out = torch.zeros(N, cfg.out_channels, self.H, self.W, **f32)
        self.d_out = torch.zeros(N, cfg.out_channels, self.H, self.W, **f32)
        self.d_ctx = torch.zeros(N * self.S, self.ctx_dim, **f32) if self.ctx_grad else None
        ctx_state = {"init": False}

        # ---- time embedding (pre-activations kept) ----
        temb_dim = boc[0] * 4
        te = m.time_embedding
        resnets = list(m._iter_resnets())
        tp_w = flat.span([r.time_emb_proj.weight for _, r in resnets], "wb")
        tp_b = flat.span([r.time_emb_proj.bias for _, r in resnets], "master")
        tp_off, n_tp = m._tproj_offsets()
        t_sin = torch.empty(N, boc[0], **f32)
        t_h1 = torch.empty(N, temb_dim, **f32)      # linear_1 output, pre-SiLU
        t_emb = torch.empty(N, temb_dim, **f32)     # linear_2 output (the SiLU lives in each time_emb_proj)
        self.tproj = torch.empty(N, n_tp, **f32)
        self.d_tproj = torch.zeros(N, n_tp, **f32)
        Fp.append(lambda: ops.timestep_embedding(self.in_t, boc[0], out=t_sin))
        Fp.append(lambda: ops.small_linear(t_sin, self.Wb(te.linear_1.weight), self.P(te.linear_1.bias), out=t_h1))
        Fp.append(lambda: ops.small_linear(t_h1, self.Wb(te.linear_2.weight), self.P(te.linear_2.bias), silu_in=True, out=t_emb))
        Fp.append(lambda: ops.small_linear(t_emb, tp_w, tp_b, silu_in=True, out=self.tproj))

        self.attn_ws = torch.empty(ops.attention_workspace_bytes(N, heads, self.H * self.W, max(boc[0] // heads, 8)) + 256,
                                   dtype=torch.uint8, device=dev)
        self.attn_bwd_ws = torch.empty(ops.attention_bwd_workspace_bytes(N, heads, self.H * self.W) + 256,
                                       dtype=torch.uint8, device=dev)

        blocks = []   # backward builders, run in reverse

        # ---- forward builders; each registers its backward as a closure over the saved tensors ----
        def resnet(prefix, r, x, skip, h, w):
            M, hw = N * h * w, h * w
            cin, cout = r.cin, r.cout
            has_sc = hasattr(r, "conv_shortcut")
            t1 = self._new(M, cin)
            raw = self._new(M, cin) if has_sc else None
            st1, st2 = torch.empty(N, 32, 2, **f32), torch.empty(N, 32, 2, **f32)   # GroupNorm (mean, rstd), kept for the backward
            self.groupnorm(Fp, x, skip, self.P(r.norm1.weight), self.P(r.norm1.bias), t1, N, hw, eps, True, raw_out=raw, stats_out=st1)
            hbuf = self._new(M, cout, F32)
            rb = (self.tproj.data_ptr() + tp_off[prefix] * 4, n_tp, hw)
            self.gemm(Fp, t1, self.Wb(r.conv1.weight), hbuf, bias=self.P(r.conv1.bias), conv=(N, h, w), rowbias_ptr=rb, gn_hw=hw)
            t2 = self._new(M, cout)
            self.groupnorm(Fp, hbuf, None, self.P(r.norm2.weight), self.P(r.norm2.bias), t2, N, hw, eps, True, stats_out=st2)
            if has_sc:
                sc = self._new(M, cout, F32)
                self.gemm(Fp, raw, self.Wb(r.conv_shortcut.weight), sc, bias=self.P(r.conv_shortcut.bias))
            else:
                sc = x
            y = self._new(M, cout, F32)
            self.gemm(Fp, t2, self.Wb(r.conv2.weight), y, bias=self.P(r.conv2.bias), residual=sc, conv=(N, h, w), gn_hw=hw)

            def backward():
                pool = self.pool
                dy = self._grad_ready(y)
                dy16 = self._prep(dy, bias_param=r.conv2.bias if tw else None)
                self.wgrad(Bp, dy16, t2, self.G(r.conv2.weight), conv=(N, h, w))
                dt2 = pool.get(M, cout)
                self.dgrad(Bp, dy16, self.Wb(r.conv2.weight), dt2, conv=(N, h, w))
                dh16 = pool.get(M, cout)
                Bp.append(lambda: ops.groupnorm_silu_bwd(hbuf, None, self.P(r.norm2.weight), self.P(r.norm2.bias), dt2, dh16, None, N, hw,
                                                         dgamma=self.G(r.norm2.weight), dbeta=self.G(r.norm2.bias), eps=eps, silu=True,
                                                         mean_rstd=st2))
                pool.put(dt2)
                # time-embedding gradient: per-image column sums of dh (conv1.bias gets the same sums, folded at the end)
                dtp = self.d_tproj.view(-1)[tp_off[prefix]:]
                Bp.append(lambda: ops.grad_prep(dh16, None, dtp, rows_per_image=hw, ldcs=n_tp))
                if tw:   # conv1.bias is added at the same place as the time embedding: its gradient is the sum over images
                    Bp.append(lambda: ops.grad_prep(dtp, None, self.G(r.conv1.bias), rows=N, N=cout, ld=n_tp))
                self.wgrad(Bp, dh16, t1, self.G(r.conv1.weight), conv=(N, h, w))
                dt1 = pool.get(M, cin)
                self.dgrad(Bp, dh16, self.Wb(r.conv1.weight), dt1, conv=(N, h, w))
                pool.put(dh16)
                if has_sc:
                    if tw:
                        Bp.append(lambda: ops.grad_prep(dy, None, self.G(r.conv_shortcut.bias)))
                    self.wgrad(Bp, dy16, raw, self.G(r.conv_shortcut.weight))
                    add = pool.get(M, cin, F32)
                    self.dgrad(Bp, dy16, self.Wb(r.conv_shortcut.weight), add)
                else:
                    add = dy
                gx, accx = self._grad_of(x)
                gs, accs = self._grad_of(skip) if skip is not None else (None, False)
                Bp.append(lambda: ops.groupnorm_silu_bwd(x, skip, self.P(r.norm1.weight), self.P(r.norm1.bias), dt1, gx, gs, N, hw, add_src=add,
                                                         acc0=accx, acc1=accs, dgamma=self.G(r.norm1.weight),
                                                         dbeta=self.G(r.norm1.bias), eps=eps, silu=True, mean_rstd=st1))
                pool.put(dt1, dy16 if dy16 is not dy else None, add if add is not dy else None)

            blocks.append((backward, r.norm1.weight))
            return y

        def xformer(prefix, a, x, h, w):
            blk = a.transformer_blocks[0]
            Cc = a.ch
            M, hw = N * h * w, h * w
            d = Cc // heads
            scale = d ** -0.5
            S = self.S
            a1m, a2m, ff = blk.attn1, blk.attn2, blk.ff
            w_qkv = flat.span([a1m.to_q.weight, a1m.to_k.weight, a1m.to_v.weight], "wb")
            w_kv2 = flat.span([a2m.to_k.weight, a2m.to_v.weight], "wb")
            t = self._new(M, Cc)
            st = torch.empty(N, 32, 2, **f32)
            self.groupnorm(Fp, x, None, self.P(a.norm.weight), self.P(a.norm.bias), t, N, hw, 1e-6, False, stats_out=st)
            hs0 = self._new(M, Cc, F32)
            self.gemm(Fp, t, self.Wb(a.proj_in.weight), hs0, bias=self.P(a.proj_in.bias))
            # self attention
            n1 = self._new(M, Cc)
            Fp.append(lambda: ops.layernorm(hs0, self.P(blk.norm1.weight), self.P(blk.norm1.bias), n1))
            qkv = self._new(M, 3 * Cc)
            self.gemm(Fp, n1, w_qkv, qkv)
            at1 = self._new(M, Cc)
            lse1 = torch.empty(N, heads, hw, **f32)
            Fp.append(lambda: ops.attention_lse(qkv, qkv, qkv, at1, lse1, N, heads, hw, hw, d, scale, ldq=3 * Cc, ldk=3 * Cc,
                                                ldv=3 * Cc, ldo=Cc, k_off=Cc, v_off=2 * Cc, ws=self.attn_ws))
            hs1 = self._new(M, Cc, F32)
            self.gemm(Fp, at1, self.Wb(a1m.to_out[0].weight), hs1, bias=self.P(a1m.to_out[0].bias), residual=hs0)
            # cross attention
            n2 = self._new(M, Cc)
            Fp.append(lambda: ops.layernorm(hs1, self.P(blk.norm2.weight), self.P(blk.norm2.bias), n2))
            q2 = self._new(M, Cc)
            self.gemm(Fp, n2, self.Wb(a2m.to_q.weight), q2)
            kv = self._new(N * S, 2 * Cc)
            self.gemm(Fp, self.in_ctx, w_kv2, kv)
            at2 = self._new(M, Cc)
            lse2 = torch.empty(N, heads, hw, **f32)
            Fp.append(lambda: ops.attention_lse(q2, kv, kv, at2, lse2, N, heads, hw, S, d, scale, ldq=Cc, ldk=2 * Cc, ldv=2 * Cc,
                                                ldo=Cc, v_off=Cc, ws=self.attn_ws))
            hs2 = self._new(M, Cc, F32)
            self.gemm(Fp, at2, self.Wb(a2m.to_out[0].weight), hs2, bias=self.P(a2m.to_out[0].bias), residual=hs1)
            # GEGLU feed-forward (pre-activation kept)
            n3 = self._new(M, Cc)
            Fp.append(lambda: ops.layernorm(hs2, self.P(blk.norm3.weight), self.P(blk.norm3.bias), n3))
            u = self._new(M, 8 * Cc)
            self.gemm(Fp, n3, self.Wb(ff.net[0].proj.weight), u, bias=self.P(ff.net[0].proj.bias))
            f = self._new(M, 4 * Cc)
            Fp.append(lambda: ops.geglu_fwd(u, f))
            hs3 = self._new(M, Cc)
            self.gemm(Fp, f, self.Wb(ff.net[2].weight), hs3, bias=self.P(ff.net[2].bias), residual=hs2)
            y = self._new(M, Cc, F32)
            self.gemm(Fp, hs3, self.Wb(a.proj_out.weight), y, bias=self.P(a.proj_out.bias), residual=x, gn_hw=hw)

            def backward():
                pool = self.pool
                dy = self._grad_ready(y)
                dy16 = self._prep(dy, bias_param=a.proj_out.bias if tw else None)
                self.wgrad(Bp, dy16, hs3, self.G(a.proj_out.weight))
                dhs = pool.get(M, Cc, F32)
                self.dgrad(Bp, dy16, self.Wb(a.proj_out.weight), dhs)
                pool.put(dy16)
                # feed-forward
                g16 = self._prep(dhs, bias_param=ff.net[2].bias if tw else None)
                self.wgrad(Bp, g16, f, self.G(ff.net[2].weight))
                dff = pool.get(M, 4 * Cc)
                self.dgrad(Bp, g16, self.Wb(ff.net[2].weight), dff)
                pool.put(g16)
                du = pool.get(M, 8 * Cc)
                Bp.append(lambda: ops.geglu_bwd(u, dff, du))
                pool.put(dff)
                if tw:
                    Bp.append(lambda: ops.grad_prep(du, None, self.G(ff.net[0].proj.bias)))
                self.wgrad(Bp, du, n3, self.G(ff.net[0].proj.weight))
                dn = pool.get(M, Cc)
                self.dgrad(Bp, du, self.Wb(ff.net[0].proj.weight), dn)
                pool.put(du)
                Bp.append(lambda: ops.layernorm_bwd(hs2, self.P(blk.norm3.weight), dn, dhs, self.G(blk.norm3.weight), self.G(blk.norm3.bias)))
                # cross attention
                g16 = self._prep(dhs, bias_param=a2m.to_out[0].bias if tw else None)
                self.wgrad(Bp, g16, at2, self.G(a2m.to_out[0].weight))
                da = pool.get(M, Cc)
                self.dgrad(Bp, g16, self.Wb(a2m.to_out[0].weight), da)
                pool.put(g16)
                dq2 = pool.get(M, Cc)
                dkv = pool.get(N * S, 2 * Cc)
                Bp.append(lambda: ops.attention_bwd(q2, kv, kv, at2, da, lse2, dq2, dkv, dkv, N, heads, hw, S, d, scale, ldq=Cc,
                                                    ldk=2 * Cc, ldv=2 * Cc, lddq=Cc, lddk=2 * Cc, lddv=2 * Cc, v_off=Cc, dv_off=Cc,
                                                    ws=self.attn_bwd_ws))
                self.wgrad(Bp, dq2, n2, self.G(a2m.to_q.weight))
                self.dgrad(Bp, dq2, self.Wb(a2m.to_q.weight), dn)
                if tw:
                    self.wgrad(Bp, dkv, self.in_ctx, flat.span([a2m.to_k.weight, a2m.to_v.weight], "grad"))
                if self.ctx_grad:
                    self.dgrad(Bp, dkv, w_kv2, self.d_ctx, residual=self.d_ctx if ctx_state["init"] else None)
                    ctx_state["init"] = True
                pool.put(dq2, dkv)
                Bp.append(lambda: ops.layernorm_bwd(hs1, self.P(blk.norm2.weight), dn, dhs, self.G(blk.norm2.weight), self.G(blk.norm2.bias)))
                # self attention
                g16 = self._prep(dhs, bias_param=a1m.to_out[0].bias if tw else None)
                self.wgrad(Bp, g16, at1, self.G(a1m.to_out[0].weight))
                self.dgrad(Bp, g16, self.Wb(a1m.to_out[0].weight), da)
                pool.put(g16)
                dqkv = pool.get(M, 3 * Cc)
                Bp.append(lambda: ops.attention_bwd(qkv, qkv, qkv, at1, da, lse1, dqkv, dqkv, dqkv, N, heads, hw, hw, d, scale,
                                                    ldq=3 * Cc, ldk=3 * Cc, ldv=3 * Cc, lddq=3 * Cc, lddk=3 * Cc, lddv=3 * Cc,
                                                    k_off=Cc, v_off=2 * Cc, dk_off=Cc, dv_off=2 * Cc, ws=self.attn_bwd_ws))
                pool.put(da)
                if tw:
                    self.wgrad(Bp, dqkv, n1, flat.span([a1m.to_q.weight, a1m.to_k.weight, a1m.to_v.weight], "grad"))
                self.dgrad(Bp, dqkv, w_qkv, dn)
                pool.put(dqkv)
                Bp.append(lambda: ops.layernorm_bwd(hs0, self.P(blk.norm1.weight), dn, dhs, self.G(blk.norm1.weight), self.G(blk.norm1.bias)))
                # proj_in + GroupNorm
                g16 = self._prep(dhs, bias_param=a.proj_in.bias if tw else None)
                self.wgrad(Bp, g16, t, self.G(a.proj_in.weight))
                self.dgrad(Bp, g16, self.Wb(a.proj_in.weight), dn)
                pool.put(g16, dhs)
                gx, accx = self._grad_of(x)
                Bp.append(lambda: ops.groupnorm_silu_bwd(x, None, self.P(a.norm.weight), self.P(a.norm.bias), dn, gx, None, N, hw, add_src=dy,
                                                         acc0=accx, dgamma=self.G(a.norm.weight), dbeta=self.G(a.norm.bias),
                                                         eps=1e-6, silu=False, mean_rstd=st))
                pool.put(dn)

            blocks.append((backward, a.norm.weight))
            return y

        def downsample(_prefix, ds, x, h, w):
            Cc = x.shape[1]
            col = self._new(N * (h // 2) * (w // 2), 9 * Cc)
            Fp.append(lambda: ops.im2col_s2(x, col, N, h, w))
            y = self._new(N * (h // 2) * (w // 2), Cc, F32)
            self.gemm(Fp, col, self.Wb(ds.conv.weight), y, bias=self.P(ds.conv.bias), gn_hw=(h // 2) * (w // 2))

            def backward():
                dy = self._grad_ready(y)
                dy16 = self._prep(dy, bias_param=ds.conv.bias if tw else None)
                self.wgrad(Bp, dy16, col, self.G(ds.conv.weight))
                dcol = self.pool.get(col.shape[0], col.shape[1])
                self.dgrad(Bp, dy16, self.Wb(ds.conv.weight), dcol)
                gx, accx = self._grad_of(x)
                Bp.append(lambda: ops.col2im_s2(dcol, gx, N, h, w, accumulate=accx))
                self.pool.put(dcol, dy16)

            blocks.append((backward, ds.conv.weight))
            return y

        def upsample(_prefix, us, x, h, w):
            Cc = x.shape[1]
            up = self._new(N * 4 * h * w, Cc)
            Fp.append(lambda: ops.upsample2x(x, up, N, h, w))
            y = self._new(N * 4 * h * w, Cc, F32)
            self.gemm(Fp, up, self.Wb(us.conv.weight), y, bias=self.P(us.conv.bias), conv=(N, 2 * h, 2 * w), gn_hw=4 * h * w)

            def backward():
                dy = self._grad_ready(y)
                dy16 = self._prep(dy, bias_param=us.conv.bias if tw else None)
                self.wgrad(Bp, dy16, up, self.G(us.conv.weight), conv=(N, 2 * h, 2 * w))
                dup = self.pool.get(up.shape[0], Cc)
                self.dgrad(Bp, dy16, self.Wb(us.conv.weight), dup, conv=(N, 2 * h, 2 * w))
                gx, accx = self._grad_of(x)
                Bp.append(lambda: ops.upsample2x_bwd(dup, gx, N, h, w, accumulate=accx))
                self.pool.put(dup, dy16)

            blocks.append((backward, us.conv.weight))
            return y

        # ---- forward graph ----
        h, w = self.H, self.W
        ci_w = flat.reg(m.conv_in.weight)
        x0 = self._new(N * h * w, boc[0], F32)
        Fp.append(lambda: ops.conv_in(self.in_sample, ci_w.wf, self.P(m.conv_in.bias), x0))

        def conv_in_backward():
            if not tw:
                return
            g = self._grad_ready(x0)
            if self.W <= 64 and 64 % self.W == 0 and cfg.in_channels <= 8:
                # weight gradient on the tensor cores: the 4-channel input is padded to 8 channels (16-byte NHWC rows) and
                # read as the MN-major B operand of the conv wgrad GEMM (TMA zero-fills the rest of the 64-column box)
                cin = cfg.in_channels
                x8 = torch.zeros(N * self.H * self.W, 8, dtype=BF16, device=dev)
                dw8 = torch.zeros(boc[0], 9 * 8, dtype=F32, device=dev)
                g16 = self.pool.get(g.shape[0], g.shape[1])
                Bp.append(lambda: ops.grad_prep(g, g16, self.G(m.conv_in.bias)))
                Bp.append(lambda: x8.view(N, self.H, self.W, 8)[..., :cin].copy_(self.in_sample.permute(0, 2, 3, 1)))
                Bp.append(lambda: dw8.zero_())
                self.wgrad(Bp, g16, x8, dw8, conv=(N, self.H, self.W))
                Bp.append(lambda: ci_w.g.view(boc[0], 9, cin).add_(dw8.view(boc[0], 9, 8)[..., :cin]))
                self.pool.put(g16)
            else:
                Bp.append(lambda: ops.conv_in_wgrad(g, self.in_sample, ci_w.g))
                Bp.append(lambda: ops.grad_prep(g, None, self.G(m.conv_in.bias)))

        blocks.append((conv_in_backward, m.conv_in.weight))
        # every forward activation is saved for the backward: nothing is released
        x, h, w = m._walk(x0, h, w, resnet=resnet, xformer=xformer, downsample=downsample, upsample=upsample, release=lambda t: None)
        co_w = flat.reg(m.conv_out.weight)
        x_last = x
        t_out = self._new(N * h * w, boc[0])
        st_out = torch.empty(N, 32, 2, **f32)
        self.groupnorm(Fp, x_last, None, self.P(m.conv_norm_out.weight), self.P(m.conv_norm_out.bias), t_out, N, h * w, eps, True,
                       stats_out=st_out)
        Fp.append(lambda: ops.conv_out(t_out, co_w.wf, self.P(m.conv_out.bias), self.out))

        # ---- backward graph: head, then the blocks in reverse, then the time MLP ----
        hw = h * w
        dt_out = self.pool.get(N * hw, boc[0])
        cout = cfg.out_channels
        tc_wgrad = tw and self.W <= 64 and 64 % self.W == 0 and cout <= 8
        if tc_wgrad:
            # conv_out weight gradient on the tensor cores: d_out (NCHW, 4 channels) padded to 8-channel NHWC bf16 rows is the
            # MN-major A operand (rows 4..127 of the 128-row MMA tile are TMA zero fill)
            dy8 = torch.zeros(N * hw, 8, dtype=BF16, device=dev)
            dwo = torch.zeros(8, 9 * boc[0], dtype=F32, device=dev)
            Bp.append(lambda: dy8.view(N, h, w, 8)[..., :cout].copy_(self.d_out.permute(0, 2, 3, 1)))
            Bp.append(lambda: dwo.zero_())
            self.wgrad(Bp, dy8, t_out, dwo, conv=(N, h, w))
            Bp.append(lambda: co_w.g.add_(dwo[:cout]))
            Bp.append(lambda: self.G(m.conv_out.bias).add_(self.d_out.sum(dim=(0, 2, 3))))
        Bp.append(lambda: ops.conv_out_bwd(self.d_out, t_out, co_w.wf, dt_out, co_w.g if (tw and not tc_wgrad) else None,
                                           self.G(m.conv_out.bias) if not tc_wgrad else None))
        gx, _ = self._grad_of(x_last)
        Bp.append(lambda: ops.groupnorm_silu_bwd(x_last, None, self.P(m.conv_norm_out.weight), self.P(m.conv_norm_out.bias), dt_out, gx, None, N, hw,
                                                 dgamma=self.G(m.conv_norm_out.weight), dbeta=self.G(m.conv_norm_out.bias),
                                                 eps=eps, silu=True, mean_rstd=st_out))
        self.pool.put(dt_out)
        if tw:
            self.ready_marks.append((len(Bp), flat.reg(m.conv_norm_out.weight).off))
        for bw, first_param in reversed(blocks):
            bw()
            if tw:
                self.ready_marks.append((len(Bp), flat.reg(first_param).off))
        if tw:
            self._time_mlp_backward(t_sin, t_h1, t_emb, tp_w, resnets, tp_off, n_tp)
            self.ready_marks.append((len(Bp), 0))

    def _time_mlp_backward(self, t_sin, t_h1, t_emb, tp_w, resnets, tp_off, n_tp):
        """d_tproj [N, n_tp] (per-image sums of every resnet's dh) -> time_emb_proj / linear_2 / linear_1 gradients.
        The three small linears run on the same tcgen05 dgrad / wgrad kernels (rows = batch, zero-filled by TMA)."""
        m, N, flat, Bp, dev = self.model, self.N, self.flat, self.bwd, self.device
        te = m.time_embedding
        temb_dim = t_emb.shape[1]
        g_tpb = flat.span([r.time_emb_proj.bias for _, r in resnets], "grad")
        g_tpw = flat.span([r.time_emb_proj.weight for _, r in resnets], "grad")
        dtp16 = torch.empty(N, n_tp, dtype=BF16, device=dev)
        Bp.append(lambda: ops.grad_prep(self.d_tproj, dtp16, g_tpb))
        a_emb = torch.empty(N, temb_dim, dtype=BF16, device=dev)
        Bp.append(lambda: ops.cast_act(t_emb, a_emb, silu=True))
        self.wgrad(Bp, dtp16, a_emb, g_tpw)
        d_emb = torch.empty(N, temb_dim, dtype=F32, device=dev)
        self.dgrad(Bp, dtp16, tp_w, d_emb)
        Bp.append(lambda: ops.silu_bwd_mul(t_emb, d_emb))
        d_emb16 = torch.empty(N, temb_dim, dtype=BF16, device=dev)
        Bp.append(lambda: ops.grad_prep(d_emb, d_emb16, self.G(te.linear_2.bias)))
        a_h1 = torch.empty(N, temb_dim, dtype=BF16, device=dev)
        Bp.append(lambda: ops.cast_act(t_h1, a_h1, silu=True))
        self.wgrad(Bp, d_emb16, a_h1, self.G(te.linear_2.weight))
        d_h1 = torch.empty(N, temb_dim, dtype=F32, device=dev)
        self.dgrad(Bp, d_emb16, self.Wb(te.linear_2.weight), d_h1)
        Bp.append(lambda: ops.silu_bwd_mul(t_h1, d_h1))
        d_h116 = torch.empty(N, temb_dim, dtype=BF16, device=dev)
        Bp.append(lambda: ops.grad_prep(d_h1, d_h116, self.G(te.linear_1.bias)))
        a_sin = torch.empty(N, t_sin.shape[1], dtype=BF16, device=dev)
        Bp.append(lambda: ops.cast_act(t_sin, a_sin, silu=False))
        self.wgrad(Bp, d_h116, a_sin, self.G(te.linear_1.weight))

    # -- execution --------------------------------------------------------------------------------
    def run_forward(self, sample, timestep, ctx):
        with torch.cuda.device(self.device):
            self.flat.refresh_weights()
            self.in_sample.copy_(sample)
            if torch.is_tensor(timestep):
                self.in_t.copy_(timestep.to(device=self.device, dtype=F32).reshape(-1).expand(self.N))
            else:
                self.in_t.fill_(float(timestep))
            self.in_ctx.copy_(ctx.reshape(self.N * self.S, self.ctx_dim))
            for op in self.fwd:
                op()
            return self.out.clone()

    def run_backward(self, d_out, on_ready=None):
        """d_out (N, C, H, W) fp32 -> parameter gradients ACCUMULATED into flat.grad (and d_ctx when asked).
        on_ready(offset) is called whenever flat.grad[offset:] has become final (the backward completes the flat
        buffer from its end towards its start), which is what a bucketed gradient allreduce overlaps on."""
        with torch.cuda.device(self.device):
            self.d_out.copy_(d_out)
            self.d_tproj.zero_()
            marks = iter(self.ready_marks)
            nxt = next(marks, None)
            for i, op in enumerate(self.bwd):
                op()
                while nxt is not None and nxt[0] == i + 1:
                    if on_ready is not None:
                        on_ready(nxt[1])
                    nxt = next(marks, None)
            return self.d_ctx.view(self.N, self.S, self.ctx_dim) if self.ctx_grad else None
