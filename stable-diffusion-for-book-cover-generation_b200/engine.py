"""Static launch plan of one UNet forward for a fixed (batch, H, W, ctx_len) geometry.

The plan is a flat list of C-ABI calls over pre-allocated NHWC bf16 activation buffers (an
(N,C,H,W) tensor is stored as [N*H*W][C], which is also the transformer's (N, H*W, C) token layout,
so no permutes exist).  Buffers are recycled through a liveness-aware pool at plan-build time; at
run time nothing is allocated, so the whole plan can be captured once into a CUDA graph and
replayed (one cudaGraphLaunch per denoising step).

Data flow per block (SURVEY.md App. A.2), each arrow = one kernel:
  resnet : [x|skip] -GN+SiLU(+cat)-> t1 -conv3x3(+bias+temb)-> h -GN+SiLU-> t2
           [x|skip] -1x1 shortcut-> sc ; t2 -conv3x3(+bias+sc)-> y
  xformer: x -GN-> t -proj_in-> hs -LN-> n -QKV-> qkv -flash attn-> a -out proj(+hs)-> hs
           -LN-> n -Q-> q ; ctx -KV-> kv (hoisted: once per context) ; flash attn -> a -out proj(+hs)-> hs
           -LN-> n -FF1+GEGLU-> f -FF2(+hs)-> hs -proj_out(+x)-> y
"""
from __future__ import annotations

import torch

from . import ops
from .plan import Builder, ContextKey, Plan, Pool, capture, profile_plan, run_plan


class Engine(Builder):
    def __init__(self, model, N, H, W, S_ctx, device, io=None):
        super().__init__(device)
        self.model, self.N, self.H, self.W, self.S = model, N, H, W, S_ctx
        self._io = io           # (in_sample, in_t, out): static buffers owned by the caller (CapturedSampler)
        cfg = model.config
        self.heads = cfg.attention_head_dim
        self.ctx_dim = cfg.cross_attention_dim
        self.plan = Plan()      # main plan (per step)
        self.ctx_plan = Plan()  # context K/V projections (once per context)
        self.graph = None
        self._ctx_key = ContextKey()
        self.debug = False      # when True (eager runs only) every tapped activation is cloned
        self.debug_out = {}
        with torch.cuda.device(device):
            self._build()

    # -- plan-building helpers --------------------------------------------------------------------
    def _tap(self, name, t, h, w):
        """Debug probe: snapshot activation `t` ([N*h*w, C] NHWC) as NCHW fp32 under `name`."""
        def op():
            if self.debug:
                self.debug_out[name] = t.float().reshape(self.N, h, w, -1).permute(0, 3, 1, 2).clone()
        self.plan.append(op, "tap")

    def _build(self):
        m, Wp, N, dev = self.model, self.model._packed, self.N, self.device
        cfg = m.config
        boc = cfg.block_out_channels
        P, pool = self.plan, Pool(dev)
        self.pool = pool
        f32 = dict(dtype=torch.float32, device=dev)

        # static inputs
        if self._io is not None:
            self.in_sample, self.in_t, self.out = self._io
        else:
            self.in_sample = torch.zeros(N, cfg.in_channels, self.H, self.W, **f32)
            self.in_t = torch.zeros(N, **f32)
            self.out = torch.zeros(N, cfg.out_channels, self.H, self.W, **f32)
        self.in_ctx = torch.zeros(N * self.S, self.ctx_dim, dtype=torch.bfloat16, device=dev)

        # ---- time embedding: sinusoid -> MLP -> all 22 time_emb_proj heads in one launch ----
        temb_dim = boc[0] * 4
        t_sin = torch.empty(N, boc[0], **f32)
        t_h = torch.empty(N, temb_dim, **f32)
        t_emb = torch.empty(N, temb_dim, **f32)
        tp_off, n_tp = m._tproj_offsets()
        self.tproj = torch.empty(N, n_tp, **f32)
        te = Wp["temb"]
        P.append(lambda: ops.timestep_embedding(self.in_t, boc[0], out=t_sin), "time_embed")
        P.append(lambda: ops.small_linear(t_sin, te["w1"], te["b1"], silu_out=True, out=t_h), "time_embed")
        P.append(lambda: ops.small_linear(t_h, te["w2"], te["b2"], out=t_emb), "time_embed")
        # all 22 time_emb_proj heads at once: (N, 1280) x (19200, 1280)^T.  The CUDA-core small_linear re-reads the 49 MB of weights
        # per group of 8 batch rows (16 us at CFG batch 2, 154 us at batch 16); from 8 rows on it is one tensor-core GEMM
        # (rows beyond N are TMA zero fill) behind a SiLU + bf16 cast of the 1280-vector
        self.large_batch = N >= 8
        if self.large_batch:
            a16 = torch.empty(N, temb_dim, dtype=torch.bfloat16, device=dev)
            P.append(lambda: ops.cast_act(t_emb, a16, silu=True), "time_embed")
            self.gemm(P, a16, Wp["tproj"]["w"], self.tproj, bias=Wp["tproj"]["b"], kind="time_embed",
                      name="time_emb_proj x22 (tensor cores)")
        else:
            P.append(lambda: ops.small_linear(t_emb, Wp["tproj"]["w"], Wp["tproj"]["b"], silu_in=True, out=self.tproj), "time_embed", 0, "time_emb_proj x22")

        # scratch for the tensor-core attention (V^T of the largest self-attention), owned by this engine
        self.attn_ws = torch.empty(ops.attention_workspace_bytes(N, self.heads, self.H * self.W, boc[0] // self.heads) + 256,
                                   dtype=torch.uint8, device=dev)

        # ---- conv_in ----
        h, w = self.H, self.W
        F32 = torch.float32   # the residual stream (block inputs/outputs, hs, conv1 -> norm2) stays fp32;
        #                       bf16 appears only where a tensor is a tensor-core operand
        x = pool.get(N * h * w, boc[0], F32)
        P.append(lambda x=x: ops.conv_in(self.in_sample, Wp["conv_in"]["w"], Wp["conv_in"]["b"], x), "conv_io", 0, "conv_in")
        self._tap("conv_in", x, h, w)

        def resnet(prefix, r, x, skip, h, w):
            wr = Wp[prefix]
            M = N * h * w
            cin, cout = r.cin, r.cout
            t1 = pool.get(M, cin)
            raw = pool.get(M, cin) if "wsc" in wr else None   # bf16 copy of [x|skip]: operand of the 1x1 shortcut
            self.groupnorm(P, x, skip, wr["g1"], wr["b1"], t1, N, h * w, cfg.norm_eps, True, raw_out=raw)
            hbuf = pool.get(M, cout, F32)
            rb = (self.tproj.data_ptr() + tp_off[prefix] * 4, n_tp, h * w)
            self.gemm(P, t1, wr["w1"], hbuf, bias=wr["cb1"], conv=(N, h, w), rowbias_ptr=rb, gn_hw=h * w)
            pool.put(t1)
            t2 = pool.get(M, cout)
            self.groupnorm(P, hbuf, None, wr["g2"], wr["b2"], t2, N, h * w, cfg.norm_eps, True)
            pool.put(hbuf)
            if "wsc" in wr:
                sc = pool.get(M, cout, F32)
                self.gemm(P, raw, wr["wsc"], sc, bias=wr["bsc"])
                pool.put(raw)
            else:
                sc = x
            y = pool.get(M, cout, F32)
            self.gemm(P, t2, wr["w2"], y, bias=wr["cb2"], residual=sc, conv=(N, h, w), gn_hw=h * w)
            pool.put(t2)
            if sc is not x:
                pool.put(sc)
            self._tap(prefix, y, h, w)
            return y

        def xformer(prefix, a, x, h, w):
            wa = Wp[prefix]
            Cc = a.ch
            M = N * h * w
            d = Cc // self.heads
            scale = d ** -0.5
            # context K/V: hoisted out of the per-step plan
            kv = torch.empty(N * self.S, 2 * Cc, dtype=torch.bfloat16, device=dev)
            self.gemm(self.ctx_plan, self.in_ctx, wa["w_kv2"], kv)
            t = pool.get(M, Cc)
            self.groupnorm(P, x, None, wa["gn_g"], wa["gn_b"], t, N, h * w, 1e-6, False)
            hs = pool.get(M, Cc, F32)
            self.gemm(P, t, wa["w_in"], hs, bias=wa["b_in"])
            # self attention
            P.append(lambda: ops.layernorm(hs, wa["ln1_g"], wa["ln1_b"], t), "layernorm")
            qkv = pool.get(M, 3 * Cc)
            self.gemm(P, t, wa["w_qkv"], qkv)
            P.append(lambda: ops.attention(qkv, qkv, qkv, t, N, self.heads, h * w, h * w, d, scale, ldq=3 * Cc,
                                           ldk=3 * Cc, ldv=3 * Cc, ldo=Cc, q_off=0, k_off=Cc, v_off=2 * Cc, ws=self.attn_ws),
                     "attention", 4.0 * N * self.heads * (h * w) * (h * w) * d, f"self-attn S{h * w} d{d}")
            pool.put(qkv)
            self.gemm(P, t, wa["w_o1"], hs, bias=wa["b_o1"], residual=hs)
            # cross attention
            P.append(lambda: ops.layernorm(hs, wa["ln2_g"], wa["ln2_b"], t), "layernorm")
            q = pool.get(M, Cc)
            self.gemm(P, t, wa["w_q2"], q)
            P.append(lambda: ops.attention(q, kv, kv, t, N, self.heads, h * w, self.S, d, scale, ldq=Cc, ldk=2 * Cc,
                                           ldv=2 * Cc, ldo=Cc, k_off=0, v_off=Cc, ws=self.attn_ws),
                     "attention", 4.0 * N * self.heads * (h * w) * self.S * d, f"cross-attn S{h * w} d{d}")
            pool.put(q)
            self.gemm(P, t, wa["w_o2"], hs, bias=wa["b_o2"], residual=hs)
            # GEGLU feed-forward
            P.append(lambda: ops.layernorm(hs, wa["ln3_g"], wa["ln3_b"], t), "layernorm")
            ff = pool.get(M, 4 * Cc)
            self.gemm(P, t, wa["w_ff1"], ff, bias=wa["b_ff1"], epilogue=ops.EPI_GEGLU, block_n=wa["ff_tile"])
            # last residual add of the block: its only consumer is proj_out's A operand -> write bf16 directly
            self.gemm(P, ff, wa["w_ff2"], t, bias=wa["b_ff2"], residual=hs)
            pool.put(ff)
            y = pool.get(M, Cc, F32)
            self.gemm(P, t, wa["w_out"], y, bias=wa["b_out"], residual=x, gn_hw=h * w)
            pool.put(t)
            pool.put(hs)
            self._tap(prefix, y, h, w)
            return y

        def downsample(prefix, _s, x, h, w):
            Cc = x.shape[1]
            col = pool.get(N * (h // 2) * (w // 2), 9 * Cc)
            P.append(lambda x=x, col=col, h=h, w=w: ops.im2col_s2(x, col, N, h, w), "resample", 0, "im2col_s2")
            h, w = h // 2, w // 2
            y = pool.get(N * h * w, Cc, F32)
            self.gemm(P, col, Wp[prefix]["w"], y, bias=Wp[prefix]["b"], gn_hw=h * w)
            pool.put(col)
            self._tap(prefix, y, h, w)
            return y

        def upsample(prefix, _s, x, h, w):
            Cc = x.shape[1]
            up = pool.get(N * 4 * h * w, Cc)
            P.append(lambda x=x, up=up, h=h, w=w: ops.upsample2x(x, up, N, h, w), "resample", 0, "upsample2x")
            h, w = 2 * h, 2 * w
            y = pool.get(N * h * w, Cc, F32)
            self.gemm(P, up, Wp[prefix]["w"], y, bias=Wp[prefix]["b"], conv=(N, h, w), gn_hw=h * w)
            pool.put(up)
            self._tap(prefix, y, h, w)
            return y

        x, h, w = m._walk(x, h, w, resnet=resnet, xformer=xformer, downsample=downsample, upsample=upsample, release=pool.put)

        # ---- out ----
        wo = Wp["conv_out"]
        t = pool.get(N * h * w, boc[0])
        self.groupnorm(P, x, None, wo["g"], wo["beta"], t, N, h * w, cfg.norm_eps, True)
        if self.large_batch and boc[0] % 64 == 0 and cfg.out_channels <= 4:
            # conv_out (320 -> 4) as an implicit GEMM on the tensor cores: [x | x] . [w_hi | w_lo] per tap (fp32-accurate weights),
            # the 4 channels padded to a 32-wide tile, then bias + NHWC -> NCHW.  The CUDA-core kernel is latency-bound at CFG batch 2
            # (32 us) and stops scaling beyond (267 us at batch 16).
            tmp = pool.get(N * h * w, 32, F32)
            self.gemm(P, t, wo["w_tc"], tmp, a1=t, conv=(N, h, w), kind="conv_io", name="conv_out (tensor cores)")
            P.append(lambda tmp=tmp: ops.nhwc_bias_to_nchw(tmp, wo["b"], self.out), "conv_io", 0, "conv_out: bias + NCHW")
        else:
            P.append(lambda t=t: ops.conv_out(t, wo["w"], wo["b"], self.out), "conv_io", 0, "conv_out")
        self.activation_bytes = pool.total

    # -- execution --------------------------------------------------------------------------------
    def set_context(self, ctx):
        """Project the (constant-over-steps) text context to every cross-attention's K/V once."""
        if self._ctx_key.matches(ctx):
            return
        self.in_ctx.copy_(ctx.reshape(self.N * self.S, self.ctx_dim))
        run_plan(self.ctx_plan)
        self._ctx_key.set(ctx)

    def run(self, sample, timestep, ctx, use_graph=True):
        with torch.cuda.device(self.device):
            self.set_context(ctx)
            self.in_sample.copy_(sample)
            if torch.is_tensor(timestep):
                self.in_t.copy_(timestep.to(device=self.device, dtype=torch.float32).reshape(-1).expand(self.N))
            else:
                self.in_t.fill_(float(timestep))
            if not use_graph:
                run_plan(self.plan)
            elif self.graph is None:
                self.graph, self.kernels_per_graph = capture(self.plan)
            else:
                self.graph.replay()
            return self.out.clone()

    def profile(self, iters=5):
        """Per-launch device time of every plan entry measured INSIDE the step (see plan.profile_plan)."""
        return profile_plan(self.plan, self.device, iters)
