"""AutoencoderKL (SURVEY.md 8f N1): the diffusers 0.7.2 class surface over b200sd kernels -- image -> latent moments (encode)
and latent -> image (decode).

Reference call sites: `AutoencoderKL.from_pretrained(path, subfolder="vae")` finetune_sd.py:325-327;
`latents = vae.encode(batch["pixel_values"]).latent_dist.sample() * 0.18215` finetune_sd.py:460-462 (the VAE is frozen,
:391-395); `vae.decode(latents / 0.18215).sample` at the end of every `pipeline(...)` call, inference.py:175-176, 342-351.

Parameters keep the diffusers names and shapes (248 tensors, 83 653 863 parameters for SD v1.x) so checkpoints load with
strict=True.  encode() / decode() build (once per geometry) a static launch plan over NHWC activation buffers and replay it as a
CUDA graph.  The plan uses the UNet's kernels at C = 128 / 256 / 512: GroupNorm+SiLU, implicit-GEMM conv3x3 on the tcgen05
GEMM (image rows of 256 / 512 pixels are tiled 128 pixels at a time), 1x1 shortcuts and linears as GEMMs with bias / residual
epilogues, nearest upsample, stride-2 im2col (pad 0: the encoder's asymmetric (0,1,0,1) padding), the CUDA-core end convs.  The
mid block's single-head 512-channel attention is two tcgen05 GEMMs around a row softmax (`scores = q k^T` as a GEMM whose
"weight" operand is k; `P v` on the data-gradient mode of the kernel, which reads v MN-major, so no transpose exists);
quant_conv is folded into the encoder's conv_out at packing time (a 1x1 conv after a conv is a conv), post_quant_conv is a
4-channel kernel.  Inference only (the reference never trains the VAE); no CPU / eager fallback.
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import ops, packing
from ._lib import B200SDError
from .plan import Builder, Plan, Pool, capture, profile_plan, run_plan
from .unet import _Config, _P, _conv, _lin

SD15_VAE_CONFIG = dict(in_channels=3, out_channels=3, latent_channels=4, block_out_channels=(128, 256, 512, 512),
                       layers_per_block=2, norm_num_groups=32, act_fn="silu", sample_size=512,
                       down_block_types=("DownEncoderBlock2D",) * 4, up_block_types=("UpDecoderBlock2D",) * 4)
F32, BF16 = torch.float32, torch.bfloat16


class AutoencoderKLOutput(SimpleNamespace):
    pass


class DecoderOutput(SimpleNamespace):
    pass


class DiagonalGaussianDistribution:
    """diffusers' posterior object: `.sample(generator)`, `.mode()`, `.mean`, `.logvar`, `.std`, `.var`, `.kl()` over the
    (B, 2C, h, w) moments; sample() draws the noise with torch.randn (same call as diffusers) and combines it in one kernel."""

    def __init__(self, parameters):
        self.parameters = parameters
        self.mean, logvar = torch.chunk(parameters, 2, dim=1)
        self.logvar = torch.clamp(logvar, -30.0, 20.0)
        self.deterministic = False

    @property
    def std(self):
        return torch.exp(0.5 * self.logvar)

    @property
    def var(self):
        return torch.exp(self.logvar)

    def sample(self, generator=None):
        """mean + std * noise, the noise drawn on the generator's device (the moments' when there is none), as the pipelines
        draw their latents"""
        p = self.parameters
        dev = p.device if generator is None else generator.device
        noise = torch.randn(self.mean.shape, generator=generator, device=dev, dtype=torch.float32).to(p.device)
        out = torch.empty_like(noise)
        ops.gaussian_sample(p.float().contiguous(), noise, out)
        return out.to(p.dtype)

    def mode(self):
        return self.mean

    def kl(self):
        return 0.5 * torch.sum(self.mean ** 2 + self.var - 1.0 - self.logvar, dim=[1, 2, 3])


# ---- parameter containers (names == diffusers state-dict keys) ----------------------------------------
class _Resnet(nn.Module):
    def __init__(self, cin, cout):
        super().__init__()
        self.cin, self.cout = cin, cout
        self.norm1 = _P(weight=(cin,), bias=(cin,))
        self.conv1 = _conv(cout, cin, 3)
        self.norm2 = _P(weight=(cout,), bias=(cout,))
        self.conv2 = _conv(cout, cout, 3)
        if cin != cout:
            self.conv_shortcut = _conv(cout, cin, 1)


class _Attn(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.ch = c
        self.group_norm = _P(weight=(c,), bias=(c,))
        self.query, self.key, self.value, self.proj_attn = _lin(c, c), _lin(c, c), _lin(c, c), _lin(c, c)


class _Sampler(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = _conv(c, c, 3)


class _Block(nn.Module):
    def __init__(self, cin, cout, layers, sampler_name):
        super().__init__()
        self.resnets = nn.ModuleList(_Resnet(cin if i == 0 else cout, cout) for i in range(layers))
        if sampler_name:
            setattr(self, sampler_name, nn.ModuleList([_Sampler(cout)]))


class _Mid(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.attentions = nn.ModuleList([_Attn(c)])
        self.resnets = nn.ModuleList([_Resnet(c, c), _Resnet(c, c)])


class _Encoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        boc = cfg.block_out_channels
        self.conv_in = _conv(boc[0], cfg.in_channels, 3)
        self.down_blocks = nn.ModuleList(_Block(boc[max(i - 1, 0)], boc[i], cfg.layers_per_block,
                                                "downsamplers" if i < len(boc) - 1 else None) for i in range(len(boc)))
        self.mid_block = _Mid(boc[-1])
        self.conv_norm_out = _P(weight=(boc[-1],), bias=(boc[-1],))
        self.conv_out = _conv(2 * cfg.latent_channels, boc[-1], 3)


class _Decoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        rev = list(reversed(cfg.block_out_channels))
        self.conv_in = _conv(rev[0], cfg.latent_channels, 3)
        self.mid_block = _Mid(rev[0])
        self.up_blocks = nn.ModuleList(_Block(rev[max(i - 1, 0)], rev[i], cfg.layers_per_block + 1,
                                              "upsamplers" if i < len(rev) - 1 else None) for i in range(len(rev)))
        self.conv_norm_out = _P(weight=(rev[-1],), bias=(rev[-1],))
        self.conv_out = _conv(cfg.out_channels, rev[-1], 3)


# ---- launch plans ----------------------------------------------------------------------------------------
class _VaeEngine(Builder):
    """Plan-building blocks shared by the encoder / decoder plans."""

    def __init__(self, model, B, H, W, device):
        super().__init__(device)
        self.model, self.B, self.H, self.W = model, B, H, W
        self.plan = Plan()
        self.pool = Pool(device)
        self.graph = None
        self.groups = model.config.norm_num_groups
        with torch.cuda.device(device):
            self._build()
        self.activation_bytes = self.pool.total

    def _gn(self, x, g, b, out, hw, silu, raw_out=None):
        self.groupnorm(self.plan, x, None, g, b, out, self.B, hw, 1e-6, silu, groups=self.groups, raw_out=raw_out)

    def _resnet(self, w, x, h, wd):
        B, pool = self.B, self.pool
        M = B * h * wd
        cin, cout = w["cin"], w["cout"]
        t1 = pool.get(M, cin)
        raw = pool.get(M, cin) if "wsc" in w else None
        self._gn(x, w["g1"], w["b1"], t1, h * wd, True, raw_out=raw)
        hb = pool.get(M, cout, F32)
        self.gemm(self.plan, t1, w["w1"], hb, bias=w["cb1"], conv=(B, h, wd))
        pool.put(t1)
        t2 = pool.get(M, cout)
        self._gn(hb, w["g2"], w["b2"], t2, h * wd, True)
        pool.put(hb)
        if raw is not None:
            sc = pool.get(M, cout, F32)
            self.gemm(self.plan, raw, w["wsc"], sc, bias=w["bsc"])
            pool.put(raw)
        else:
            sc = x
        y = pool.get(M, cout, F32)
        self.gemm(self.plan, t2, w["w2"], y, bias=w["cb2"], residual=sc, conv=(B, h, wd))
        pool.put(t2)
        if sc is not x:
            pool.put(sc)
        pool.put(x)
        return y

    def _attention(self, w, x, h, wd):
        """AttentionBlock: GN -> q, k, v -> softmax(q k^T / sqrt(C)) v -> proj (+x); one head over all C channels"""
        B, pool, dev = self.B, self.pool, self.device
        S, C = h * wd, w["C"]
        M = B * S
        t = pool.get(M, C)
        self._gn(x, w["g"], w["b"], t, S, False)
        q, k, v = pool.get(M, C), pool.get(M, C), pool.get(M, C)
        self.gemm(self.plan, t, w["wq"], q, bias=w["bq"])
        self.gemm(self.plan, t, w["wk"], k, bias=w["bk"])
        self.gemm(self.plan, t, w["wv"], v, bias=w["bv"])
        scores = pool.get(S, S, F32)
        probs = pool.get(S, S)
        o = t                                          # the normalised input is dead once q, k, v exist
        scale = float(C) ** -0.5                       # (q C^-1/4) . (k C^-1/4)
        for b in range(B):
            qb, kb, vb, ob = (z[b * S:(b + 1) * S] for z in (q, k, v, o))
            self.gemm(self.plan, qb, kb, scores)                                           # scores = q k^T  (k is the "weight" operand)
            self.plan.append(lambda: ops.softmax_rows(scores, probs, scale), "attention", 0, "softmax rows")
            self.dgrad(self.plan, probs, vb, ob, name=f"attention P.v S{S} C{C}")   # out = P v  (v read MN-major: no transpose)
        y = pool.get(M, C, F32)
        self.gemm(self.plan, o, w["wo"], y, bias=w["bo"], residual=x)
        for z in (q, k, v, scores, probs, t, x):
            pool.put(z)
        return y

    def _mid(self, prefix, x, h, wd):
        W = self.model._packed
        x = self._resnet(W[prefix + ".res0"], x, h, wd)
        x = self._attention(W[prefix + ".attn"], x, h, wd)
        return self._resnet(W[prefix + ".res1"], x, h, wd)

    def profile(self, iters=3):
        return profile_plan(self.plan, self.device, iters)

    def _replay(self, set_inputs):
        with torch.cuda.device(self.device):
            set_inputs()
            if self.graph is not None:
                self.graph.replay()
            elif self.model.use_cuda_graph:
                self.graph, _ = capture(self.plan)
            else:
                run_plan(self.plan)
            return self.out.clone()


class VaeDecodeEngine(_VaeEngine):
    """latents (B, 4, h, w) -> image (B, 3, 8h, 8w)"""

    def _build(self):
        m, Wp, B, dev, P, pool = self.model, self.model._packed, self.B, self.device, self.plan, self.pool
        cfg = m.config
        rev = list(reversed(cfg.block_out_channels))
        h, w = self.H, self.W
        lc = cfg.latent_channels
        self.in_z = torch.zeros(B, lc, h, w, dtype=F32, device=dev)
        z2 = torch.zeros(B, lc, h, w, dtype=F32, device=dev)
        P.append(lambda: ops.conv1x1_small(self.in_z, Wp["post_quant"]["w"], Wp["post_quant"]["b"], z2), "conv_io", 0, "post_quant_conv")
        x = pool.get(B * h * w, rev[0], F32)
        P.append(lambda x=x: ops.conv_in(z2, Wp["dec.conv_in"]["w"], Wp["dec.conv_in"]["b"], x), "conv_io", 0, "decoder conv_in")
        x = self._mid("dec.mid", x, h, w)
        for i, blk in enumerate(m.decoder.up_blocks):
            for j in range(len(blk.resnets)):
                x = self._resnet(Wp[f"dec.up{i}.res{j}"], x, h, w)
            if hasattr(blk, "upsamplers"):
                wu = Wp[f"dec.up{i}.us"]
                C = x.shape[1]
                up = pool.get(B * 4 * h * w, C)
                P.append(lambda x=x, up=up, h=h, w=w: ops.upsample2x(x, up, B, h, w), "resample", 0, "upsample2x")
                pool.put(x)
                h, w = 2 * h, 2 * w
                x = pool.get(B * h * w, C, F32)
                self.gemm(self.plan, up, wu["w"], x, bias=wu["b"], conv=(B, h, w))
                pool.put(up)
        wo = Wp["dec.conv_out"]
        t = pool.get(B * h * w, rev[-1])
        self._gn(x, wo["g"], wo["beta"], t, h * w, True)
        self.out = torch.zeros(B, cfg.out_channels, h, w, dtype=F32, device=dev)
        # conv_out (128 -> 3) on the tensor cores: [x | x] . [w_hi | w_lo] per tap (fp32-accurate weights), the 3 channels padded
        # to a 32-wide tile, then bias + NHWC -> NCHW (the CUDA-core kernel took 0.5 ms of an 11 ms decode at 512 x 512)
        tmp = pool.get(B * h * w, 32, F32)
        self.gemm(P, t, wo["w_tc"], tmp, a1=t, conv=(B, h, w), block_n=32, kind="conv_io", name="decoder conv_out (tensor cores)")
        P.append(lambda tmp=tmp: ops.nhwc_bias_to_nchw(tmp, wo["b"], self.out), "conv_io", 0, "decoder conv_out: bias + NCHW")

    def run(self, z):
        return self._replay(lambda: self.in_z.copy_(z))


class VaeEncodeEngine(_VaeEngine):
    """image (B, 3, H, W) -> moments (B, 8, H/8, W/8) = quant_conv(encoder(x))"""

    def _build(self):
        m, Wp, B, dev, P, pool = self.model, self.model._packed, self.B, self.device, self.plan, self.pool
        cfg = m.config
        boc = cfg.block_out_channels
        h, w = self.H, self.W
        self.in_x = torch.zeros(B, 4, h, w, dtype=F32, device=dev)       # 3 image channels + a zero one (conv_in reads 4)
        x = pool.get(B * h * w, boc[0], F32)
        P.append(lambda x=x: ops.conv_in(self.in_x, Wp["enc.conv_in"]["w"], Wp["enc.conv_in"]["b"], x), "conv_io", 0, "encoder conv_in")
        for i, blk in enumerate(m.encoder.down_blocks):
            for j in range(len(blk.resnets)):
                x = self._resnet(Wp[f"enc.down{i}.res{j}"], x, h, w)
            if hasattr(blk, "downsamplers"):
                wd_ = Wp[f"enc.down{i}.ds"]
                C = x.shape[1]
                col = pool.get(B * (h // 2) * (w // 2), 9 * C)
                P.append(lambda x=x, col=col, h=h, w=w: ops.im2col_s2(x, col, B, h, w, pad=0), "resample", 0, "im2col_s2 (pad 0)")
                pool.put(x)
                h, w = h // 2, w // 2
                x = pool.get(B * h * w, C, F32)
                self.gemm(self.plan, col, wd_["w"], x, bias=wd_["b"])
                pool.put(col)
        x = self._mid("enc.mid", x, h, w)
        wo = Wp["enc.conv_out"]
        t = pool.get(B * h * w, boc[-1])
        self._gn(x, wo["g"], wo["beta"], t, h * w, True)
        tmp = pool.get(B * h * w, 32, F32)
        self.gemm(self.plan, t, wo["w_tc"], tmp, a1=t, conv=(B, h, w), block_n=32)
        self.out = torch.zeros(B, 2 * cfg.latent_channels, h, w, dtype=F32, device=dev)
        P.append(lambda tmp=tmp: ops.nhwc_bias_to_nchw(tmp, wo["b"], self.out), "conv_io", 0, "conv_out + quant_conv: bias + NCHW")

    def run(self, x):
        return self._replay(lambda: self.in_x[:, :x.shape[1]].copy_(x))


class AutoencoderKL(nn.Module):
    config_name = "config.json"

    def __init__(self, **kw):
        super().__init__()
        cfg = dict(SD15_VAE_CONFIG)
        unknown = set(kw) - set(cfg)
        if unknown:
            raise TypeError(f"AutoencoderKL: unexpected config keys {sorted(unknown)}")
        cfg.update(kw)
        cfg["block_out_channels"] = tuple(cfg["block_out_channels"])
        if any(c % 64 for c in cfg["block_out_channels"]):
            raise ValueError("block_out_channels must be multiples of 64")
        if cfg["in_channels"] > 4 or cfg["out_channels"] > 4 or cfg["latent_channels"] != 4:
            raise NotImplementedError("image channels <= 4 and 4 latent channels (the SD v1.x VAE)")
        if cfg["act_fn"] != "silu":
            raise NotImplementedError("act_fn must be 'silu'")
        self.config = _Config(cfg)
        c = self.config
        self.encoder, self.decoder = _Encoder(c), _Decoder(c)
        self.quant_conv = _conv(2 * c.latent_channels, 2 * c.latent_channels, 1)
        self.post_quant_conv = _conv(c.latent_channels, c.latent_channels, 1)
        self.use_cuda_graph = True
        self._packed, self._engines, self._param_versions = None, {}, None
        self.reset_parameters()

    @torch.no_grad()
    def reset_parameters(self):
        """torch-default init (kaiming-uniform for conv / linear, ones / zeros for norms)"""
        params = dict(self.named_parameters())
        for name, p in params.items():
            is_norm = "norm" in name.rsplit(".", 2)[-2]
            if name.endswith("weight"):
                if is_norm:
                    p.fill_(1.0)
                else:
                    p.uniform_(-(1.0 / p[0].numel()) ** 0.5, (1.0 / p[0].numel()) ** 0.5)
            elif is_norm:
                p.zero_()
            else:
                w = params[name[:-4] + "weight"]
                p.uniform_(-(1.0 / w[0].numel()) ** 0.5, (1.0 / w[0].numel()) ** 0.5)

    @property
    def device(self):
        return self.quant_conv.weight.device

    @property
    def dtype(self):
        return self.quant_conv.weight.dtype

    def _apply(self, fn, *a, **kw):
        r = super()._apply(fn, *a, **kw)
        self._packed, self._engines = None, {}
        return r

    def load_state_dict(self, *a, **kw):
        r = super().load_state_dict(*a, **kw)
        self._packed, self._engines = None, {}
        return r

    # -- (de)serialisation (diffusers directory layout) ---------------------------------------------------
    @classmethod
    def from_pretrained(cls, path, subfolder=None, torch_dtype=None, **kw):
        d = path if subfolder is None else os.path.join(path, subfolder)
        with open(os.path.join(d, cls.config_name)) as f:
            cfg = json.load(f)
        model = cls(**{k: v for k, v in cfg.items() if k in SD15_VAE_CONFIG})
        st_path, bin_path = os.path.join(d, "diffusion_pytorch_model.safetensors"), os.path.join(d, "diffusion_pytorch_model.bin")
        if os.path.exists(st_path):
            from safetensors.torch import load_file
            sd = load_file(st_path)
        elif os.path.exists(bin_path):
            sd = torch.load(bin_path, map_location="cpu")
        else:
            raise FileNotFoundError(f"no diffusion_pytorch_model.(safetensors|bin) under {d}")
        model.load_state_dict(sd, strict=True)
        if torch_dtype is not None:
            model.to(dtype=torch_dtype)
        return model.eval()

    def save_pretrained(self, path, safe_serialization=False):
        os.makedirs(path, exist_ok=True)
        with open(os.path.join(path, self.config_name), "w") as f:
            json.dump(dict(self.config, _class_name="AutoencoderKL", _diffusers_version="0.7.2"), f, indent=2)
        sd = {k: v.detach().cpu().contiguous() for k, v in self.state_dict().items()}
        if safe_serialization:
            from safetensors.torch import save_file
            save_file(sd, os.path.join(path, "diffusion_pytorch_model.safetensors"))
        else:
            torch.save(sd, os.path.join(path, "diffusion_pytorch_model.bin"))

    # -- weight packing ---------------------------------------------------------------------------------------
    @torch.no_grad()
    def _pack_weights(self):
        W = {}
        f32 = lambda t: t.detach().float().contiguous().clone()
        cfg = self.config

        def res(prefix, r):
            W[prefix] = dict(cin=r.cin, cout=r.cout, g1=f32(r.norm1.weight), b1=f32(r.norm1.bias),
                             w1=packing.pack_conv3x3(r.conv1.weight.detach().float()), cb1=f32(r.conv1.bias),
                             g2=f32(r.norm2.weight), b2=f32(r.norm2.bias),
                             w2=packing.pack_conv3x3(r.conv2.weight.detach().float()), cb2=f32(r.conv2.bias))
            if hasattr(r, "conv_shortcut"):
                W[prefix]["wsc"] = packing.pack_linear(r.conv_shortcut.weight.detach().float())
                W[prefix]["bsc"] = f32(r.conv_shortcut.bias)

        def mid(prefix, mb):
            res(prefix + ".res0", mb.resnets[0])
            res(prefix + ".res1", mb.resnets[1])
            a = mb.attentions[0]
            lin = lambda l: packing.pack_linear(l.weight.detach().float())
            W[prefix + ".attn"] = dict(C=a.ch, g=f32(a.group_norm.weight), b=f32(a.group_norm.bias), wq=lin(a.query), bq=f32(a.query.bias),
                                       wk=lin(a.key), bk=f32(a.key.bias), wv=lin(a.value), bv=f32(a.value.bias),
                                       wo=lin(a.proj_attn), bo=f32(a.proj_attn.bias))

        def conv_in4(conv):
            """[Cout][9][4] fp32 for the CUDA-core conv_in kernel (3-channel images get a zero fourth input channel)"""
            w = conv.weight.detach().float()
            if w.shape[1] < 4:
                w = torch.cat([w, w.new_zeros(w.shape[0], 4 - w.shape[1], 3, 3)], dim=1)
            return dict(w=packing.pack_conv3x3_f32(w), b=f32(conv.bias))

        enc, dec = self.encoder, self.decoder
        W["enc.conv_in"] = conv_in4(enc.conv_in)
        for i, b in enumerate(enc.down_blocks):
            for j, r in enumerate(b.resnets):
                res(f"enc.down{i}.res{j}", r)
            if hasattr(b, "downsamplers"):
                c = b.downsamplers[0].conv
                W[f"enc.down{i}.ds"] = dict(w=packing.pack_conv3x3(c.weight.detach().float()), b=f32(c.bias))
        mid("enc.mid", enc.mid_block)
        # quant_conv o conv_out: W'[o] = sum_m Wq[o][m] Wc[m], b' = Wq bc + bq (a 1x1 conv after a conv is a conv); the 8 output
        # channels are zero-padded to a 32-wide tensor-core tile
        wq = self.quant_conv.weight.detach().float().reshape(2 * cfg.latent_channels, 2 * cfg.latent_channels)
        wc = torch.einsum("om,mikl->oikl", wq, enc.conv_out.weight.detach().float())
        bc = wq @ enc.conv_out.bias.detach().float() + self.quant_conv.bias.detach().float()
        # [x | x] . [w_hi | w_lo] per tap keeps the fp32 weights of this last layer to ~2^-17 (as the UNet's conv_out does)
        w_tc = packing.pack_conv_out_tc(wc, pad_to=32)
        W["enc.conv_out"] = dict(g=f32(enc.conv_norm_out.weight), beta=f32(enc.conv_norm_out.bias), w_tc=w_tc, b=bc.contiguous())
        pq = self.post_quant_conv
        W["post_quant"] = dict(w=f32(pq.weight).reshape(pq.weight.shape[0], -1).contiguous(), b=f32(pq.bias))
        W["dec.conv_in"] = conv_in4(dec.conv_in)
        mid("dec.mid", dec.mid_block)
        for i, b in enumerate(dec.up_blocks):
            for j, r in enumerate(b.resnets):
                res(f"dec.up{i}.res{j}", r)
            if hasattr(b, "upsamplers"):
                c = b.upsamplers[0].conv
                W[f"dec.up{i}.us"] = dict(w=packing.pack_conv3x3(c.weight.detach().float()), b=f32(c.bias))
        W["dec.conv_out"] = dict(g=f32(dec.conv_norm_out.weight), beta=f32(dec.conv_norm_out.bias),
                                 w_tc=packing.pack_conv_out_tc(dec.conv_out.weight.detach().float(), pad_to=32), b=f32(dec.conv_out.bias))
        self._packed = W
        self._param_versions = self._versions()

    def _versions(self):
        ps = self.__dict__.get("_param_list")
        if ps is None:
            ps = self.__dict__["_param_list"] = list(self.parameters())
        return sum(p._version for p in ps)

    def _engine(self, kind, B, H, W, dev):
        if not dev.type == "cuda":
            raise B200SDError("b200sd.AutoencoderKL runs on CUDA only (no CPU fallback)")
        if self._packed is None or self._versions() != self._param_versions:
            with torch.cuda.device(dev):
                self._pack_weights()
            self._engines = {}
        key = (kind, B, H, W, dev.index)
        eng = self._engines.get(key)
        if eng is None:
            if len(self._engines) >= 4:
                self._engines.clear()          # each engine owns its activation buffers (GBs at 512 x 512)
            eng = self._engines[key] = (VaeDecodeEngine if kind == "dec" else VaeEncodeEngine)(self, B, H, W, dev)
        return eng

    # -- the diffusers surface --------------------------------------------------------------------------------
    @torch.no_grad()
    def encode(self, x, return_dict: bool = True):
        n_down = len(self.config.block_out_channels) - 1
        if x.dim() != 4 or x.shape[1] != self.config.in_channels:
            raise ValueError(f"sample must be (B, {self.config.in_channels}, H, W), got {tuple(x.shape)}")
        B, _, H, W = x.shape
        if H % (1 << n_down) or W % (1 << n_down):
            raise ValueError(f"H and W must be multiples of {1 << n_down}")
        if W > 128 and W % 128:
            raise NotImplementedError("image widths above 128 must be multiples of 128")
        moments = self._engine("enc", B, H, W, x.device).run(x.float())
        post = DiagonalGaussianDistribution(moments.to(x.dtype))
        return AutoencoderKLOutput(latent_dist=post) if return_dict else (post,)

    @torch.no_grad()
    def decode(self, z, return_dict: bool = True):
        if z.dim() != 4 or z.shape[1] != self.config.latent_channels:
            raise ValueError(f"latents must be (B, {self.config.latent_channels}, h, w), got {tuple(z.shape)}")
        B, _, h, w = z.shape
        n_up = len(self.config.block_out_channels) - 1
        if (w << n_up) > 128 and (w << n_up) % 128:
            raise NotImplementedError("image widths above 128 must be multiples of 128")
        img = self._engine("dec", B, h, w, z.device).run(z.float()).to(z.dtype)
        return DecoderOutput(sample=img) if return_dict else (img,)

    def forward(self, sample, sample_posterior: bool = False, return_dict: bool = True, generator=None):
        post = self.encode(sample).latent_dist
        z = post.sample(generator=generator) if sample_posterior else post.mode()
        return self.decode(z, return_dict=return_dict)
