"""UNet2DConditionModel facade: the diffusers 0.7.2 class surface (SURVEY.md 8b) over the sm_100a
kernels.

    unet(noisy_latents, timesteps, encoder_hidden_states).sample            finetune_sd.py:480-481
    UNet2DConditionModel.from_pretrained(path, subfolder="unet")            finetune_sd.py:328-330
    unet.in_channels / .config / .to() / .parameters() / .eval() / ...      finetune_sd.py:198, 393-395

Parameters keep the diffusers names and shapes (686 tensors, App. A.4) so SD v1.x checkpoints load
with strict=True.  forward() does not run torch modules: it builds (once per input geometry) a static
launch plan over NHWC bf16 activation buffers -- every entry is one C-ABI call into libb200sd.so --
and replays it, optionally as a CUDA graph.  There is no eager / CPU fallback.
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import ops, packing
from ._lib import B200SDError

SD15_CONFIG = dict(
    sample_size=64, in_channels=4, out_channels=4, center_input_sample=False, flip_sin_to_cos=True, freq_shift=0,
    down_block_types=("CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "DownBlock2D"),
    up_block_types=("UpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D"),
    block_out_channels=(320, 640, 1280, 1280), layers_per_block=2, downsample_padding=1, mid_block_scale_factor=1,
    act_fn="silu", norm_num_groups=32, norm_eps=1e-5, cross_attention_dim=768, attention_head_dim=8,
)


class UNet2DConditionOutput(SimpleNamespace):
    pass


class _Config(dict):
    """dict with attribute access (diffusers' FrozenDict behaves like this)."""
    __getattr__ = dict.__getitem__


# ---------------------------------------------------------------------------------------------
# parameter containers (names == diffusers state-dict keys; they hold no forward logic)
# ---------------------------------------------------------------------------------------------
class _P(nn.Module):
    def __init__(self, **shapes):
        super().__init__()
        for name, shape in shapes.items():
            self.register_parameter(name, nn.Parameter(torch.empty(shape)))


def _conv(cout, cin, k):
    return _P(weight=(cout, cin, k, k), bias=(cout,))


def _lin(cout, cin, bias=True):
    return _P(weight=(cout, cin), bias=(cout,)) if bias else _P(weight=(cout, cin))


def _norm(c):
    return _P(weight=(c,), bias=(c,))


def _resnet(cin, cout, temb):
    m = nn.Module()
    m.norm1, m.conv1, m.time_emb_proj = _norm(cin), _conv(cout, cin, 3), _lin(cout, temb)
    m.norm2, m.conv2 = _norm(cout), _conv(cout, cout, 3)
    if cin != cout:
        m.conv_shortcut = _conv(cout, cin, 1)
    m.cin, m.cout = cin, cout
    return m


def _attn(dim, ctx_dim):
    m = nn.Module()
    m.to_q, m.to_k, m.to_v = _lin(dim, dim, False), _lin(dim, ctx_dim, False), _lin(dim, ctx_dim, False)
    m.to_out = nn.ModuleList([_lin(dim, dim)])
    return m


def _xformer(ch, ctx_dim):
    m = nn.Module()
    m.norm, m.proj_in, m.proj_out = _norm(ch), _conv(ch, ch, 1), _conv(ch, ch, 1)
    blk = nn.Module()
    blk.attn1, blk.attn2 = _attn(ch, ch), _attn(ch, ctx_dim)
    blk.norm1, blk.norm2, blk.norm3 = _norm(ch), _norm(ch), _norm(ch)
    ff = nn.Module()
    geglu = nn.Module()
    geglu.proj = _lin(ch * 8, ch)
    ff.net = nn.ModuleList([geglu, nn.Identity(), _lin(ch, ch * 4)])
    blk.ff = ff
    m.transformer_blocks = nn.ModuleList([blk])
    m.ch = ch
    return m


def _sampler(ch):
    m = nn.Module()
    m.conv = _conv(ch, ch, 3)
    return m


class UNet2DConditionModel(nn.Module):
    config_name = "config.json"

    def __init__(self, **overrides):
        super().__init__()
        cfg = dict(SD15_CONFIG)
        unknown = set(overrides) - set(cfg) - {"_class_name", "_diffusers_version", "_name_or_path"}
        if unknown:
            raise TypeError(f"UNet2DConditionModel: unexpected config keys {sorted(unknown)}")
        cfg.update({k: v for k, v in overrides.items() if k in cfg})
        for k in ("down_block_types", "up_block_types", "block_out_channels"):
            cfg[k] = tuple(cfg[k])
        self.config = _Config(cfg)
        boc = cfg["block_out_channels"]
        if cfg["act_fn"] != "silu" or cfg["norm_num_groups"] != 32 or cfg["center_input_sample"]:
            raise NotImplementedError("only the SD v1.x UNet configuration family is supported")
        if any(c % 64 for c in boc):
            raise NotImplementedError("block_out_channels must be multiples of 64 (tensor-core tile K)")
        self.in_channels = cfg["in_channels"]
        temb = boc[0] * 4
        ctx = cfg["cross_attention_dim"]
        L = cfg["layers_per_block"]

        self.conv_in = _conv(boc[0], cfg["in_channels"], 3)
        te = nn.Module()
        te.linear_1, te.linear_2 = _lin(temb, boc[0]), _lin(temb, temb)
        self.time_embedding = te

        self.down_blocks = nn.ModuleList()
        out_ch = boc[0]
        for i, typ in enumerate(cfg["down_block_types"]):
            in_ch, out_ch = out_ch, boc[i]
            b = nn.Module()
            b.resnets = nn.ModuleList([_resnet(in_ch if j == 0 else out_ch, out_ch, temb) for j in range(L)])
            if typ.startswith("CrossAttn"):
                b.attentions = nn.ModuleList([_xformer(out_ch, ctx) for _ in range(L)])
            if i != len(boc) - 1:
                b.downsamplers = nn.ModuleList([_sampler(out_ch)])
            self.down_blocks.append(b)

        mid = nn.Module()
        mid.attentions = nn.ModuleList([_xformer(boc[-1], ctx)])
        mid.resnets = nn.ModuleList([_resnet(boc[-1], boc[-1], temb), _resnet(boc[-1], boc[-1], temb)])
        self.mid_block = mid

        self.up_blocks = nn.ModuleList()
        rev = list(reversed(boc))
        out_ch = rev[0]
        for i, typ in enumerate(cfg["up_block_types"]):
            prev, out_ch = out_ch, rev[i]
            in_ch = rev[min(i + 1, len(boc) - 1)]
            b = nn.Module()
            res = []
            for j in range(L + 1):
                skip = in_ch if j == L else out_ch
                rin = prev if j == 0 else out_ch
                r = _resnet(rin + skip, out_ch, temb)
                r.c_x, r.c_skip = rin, skip
                res.append(r)
            b.resnets = nn.ModuleList(res)
            if typ.startswith("CrossAttn"):
                b.attentions = nn.ModuleList([_xformer(out_ch, ctx) for _ in range(L + 1)])
            if i != len(boc) - 1:
                b.upsamplers = nn.ModuleList([_sampler(out_ch)])
            self.up_blocks.append(b)

        self.conv_norm_out = _norm(boc[0])
        self.conv_out = _conv(cfg["out_channels"], boc[0], 3)

        self.reset_parameters()
        self._engines = {}
        self._packed = None
        self._dirty = True
        self.use_cuda_graph = True
        self._gradient_checkpointing = False
        self._flat = None            # train.FlatParams (flat bf16 weights + flat fp32 gradients), built on first training call
        self._train_engines = {}
        self._direct_grads = False
        self._precision = "bf16"       # "bf16" (tensor-core operands rounded to bf16) | "fp32" (split-bf16 3-term products, engine_fp32.py)
        self._grad_ready_hook = None   # direct mode: called with `offset` when flat_gradients()[offset:] is final (trainer.py)

    # -- init / (de)serialisation ---------------------------------------------------------------
    @torch.no_grad()
    def reset_parameters(self):
        """torch-default init (kaiming-uniform a=sqrt(5) for conv/linear, ones/zeros for norms)."""
        params = dict(self.named_parameters())
        for name, p in params.items():
            leaf = name.rsplit(".", 2)
            is_norm = "norm" in leaf[-2]
            if name.endswith("weight"):
                if is_norm:
                    p.fill_(1.0)
                else:
                    fan_in = p[0].numel()
                    bound = (1.0 / fan_in) ** 0.5
                    p.uniform_(-bound, bound)
            else:
                if is_norm:
                    p.zero_()
                else:
                    w = params[name[:-4] + "weight"]
                    bound = (1.0 / w[0].numel()) ** 0.5
                    p.uniform_(-bound, bound)

    @classmethod
    def from_config(cls, cfg):
        return cls(**{k: v for k, v in dict(cfg).items() if not k.startswith("_")})

    @classmethod
    def from_pretrained(cls, path, subfolder=None, torch_dtype=None, **kw):
        d = path if subfolder is None else os.path.join(path, subfolder)
        with open(os.path.join(d, cls.config_name)) as f:
            cfg = json.load(f)
        model = cls(**{k: v for k, v in cfg.items() if not k.startswith("_")})
        st_path = os.path.join(d, "diffusion_pytorch_model.safetensors")
        bin_path = os.path.join(d, "diffusion_pytorch_model.bin")
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
        cfg = dict(self.config, _class_name="UNet2DConditionModel", _diffusers_version="0.7.2")
        with open(os.path.join(path, self.config_name), "w") as f:
            json.dump(cfg, f, indent=2)
        # .contiguous(): after a training call the parameters are (possibly permuted) views of the flat master buffer
        sd = {k: v.detach().cpu().contiguous() for k, v in self.state_dict().items()}
        if safe_serialization:
            from safetensors.torch import save_file
            save_file(sd, os.path.join(path, "diffusion_pytorch_model.safetensors"))
        else:
            torch.save(sd, os.path.join(path, "diffusion_pytorch_model.bin"))

    def load_state_dict(self, *a, **kw):
        r = super().load_state_dict(*a, **kw)
        self._dirty = True
        return r

    def _apply(self, fn, *a, **kw):
        r = super()._apply(fn, *a, **kw)
        self._dirty = True
        self._engines = {}
        self._flat = None
        self._train_engines = {}
        self._rehome()
        return r

    def _rehome(self):
        """As soon as the fp32 parameters sit on a GPU, move them into the flat kernel-layout master buffer (train.FlatParams:
        every Parameter becomes a view of it; 3x3 conv weights permuted views).  Doing this at .to(device) time -- not lazily at
        the first training forward -- matters for wrappers that record the parameters' strides when they are constructed:
        DistributedDataParallel (accelerator.prepare, finetune_sd.py:363, 386) builds its gradient buckets from them, and
        gradients whose strides differ from what it saw come back corrupted (found by tests/test_dropin_gpu.py)."""
        ps = list(self.parameters())
        if not ps or any((not p.is_cuda) or p.dtype != torch.float32 or p.device != ps[0].device for p in ps):
            return
        from .train import FlatParams
        with torch.cuda.device(ps[0].device):
            self._flat = FlatParams(self, ps[0].device, lazy=True)

    def set_precision(self, precision: str):
        """"bf16": the fast plan (noise prediction within 1e-2 of the fp32 reference).  "fp32": the accuracy plan
        (engine_fp32.py: every contraction as a 3-term split-bf16 product with fp32 accumulation, fp32 attention /
        norms / GEGLU; within 1e-4).  Inference only; training always runs the bf16 plan on fp32 master weights."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        if precision != self._precision:
            self._precision = precision
            self._engines = {}
        return self

    def enable_direct_gradients(self, enabled: bool = True):
        """param.grad become views of ONE flat fp32 gradient buffer that the backward kernels accumulate into
        (see autograd.py).  Use `flat_gradients()` for bucketed allreduce / a fused optimizer."""
        self._direct_grads = bool(enabled)
        return self

    def flat_gradients(self):
        """the flat fp32 gradient buffer (kernel layout) -- None before the first training forward"""
        return None if self._flat is None else self._flat.grad

    def zero_grad(self, set_to_none: bool = True):
        if self._direct_grads and self._flat is not None and self._flat.grad is not None:
            self._flat.zero_grad()
            self._flat.attach_grads()
            return
        super().zero_grad(set_to_none=set_to_none)

    def mark_weights_changed(self):
        """The inference engines hold their own packed bf16 copy of the weights: call this after changing parameters through
        anything that bumps no tensor version (raw kernels; b200sd.trainer.FlatAdamW does it itself)."""
        self._dirty = True

    @property
    def device(self):
        return self.conv_in.weight.device

    @property
    def dtype(self):
        return self.conv_in.weight.dtype

    def enable_gradient_checkpointing(self):
        """accepted for API compatibility (finetune_sd.py:389); activations of one step fit in HBM3e (180 GB) and are kept"""
        self._gradient_checkpointing = True

    # -- weight packing -------------------------------------------------------------------------
    @torch.no_grad()
    def _pack_weights(self):
        """diffusers layouts -> kernel layouts (bf16 K-major GEMM operands, fp32 biases / norms)."""
        W = {}
        f32 = lambda t: t.detach().float().clone()     # a COPY: FlatParams later re-homes the parameter storage

        def res(prefix, r):
            W[prefix] = dict(
                g1=f32(r.norm1.weight), b1=f32(r.norm1.bias), w1=packing.pack_conv3x3(r.conv1.weight.detach()),
                cb1=f32(r.conv1.bias), g2=f32(r.norm2.weight), b2=f32(r.norm2.bias),
                w2=packing.pack_conv3x3(r.conv2.weight.detach()), cb2=f32(r.conv2.bias))
            if hasattr(r, "conv_shortcut"):
                W[prefix]["wsc"] = packing.pack_linear(r.conv_shortcut.weight.detach())
                W[prefix]["bsc"] = f32(r.conv_shortcut.bias)

        def xf(prefix, a):
            blk = a.transformer_blocks[0]
            C = a.ch
            tile = ops.geglu_tile(8 * C)
            wg, bg = packing.pack_geglu(blk.ff.net[0].proj.weight.detach().float(), blk.ff.net[0].proj.bias.detach().float(), tile)
            W[prefix] = dict(
                gn_g=f32(a.norm.weight), gn_b=f32(a.norm.bias),
                w_in=packing.pack_linear(a.proj_in.weight.detach()), b_in=f32(a.proj_in.bias),
                w_out=packing.pack_linear(a.proj_out.weight.detach()), b_out=f32(a.proj_out.bias),
                ln1_g=f32(blk.norm1.weight), ln1_b=f32(blk.norm1.bias),
                ln2_g=f32(blk.norm2.weight), ln2_b=f32(blk.norm2.bias),
                ln3_g=f32(blk.norm3.weight), ln3_b=f32(blk.norm3.bias),
                w_qkv=packing.pack_linear(torch.cat([blk.attn1.to_q.weight, blk.attn1.to_k.weight, blk.attn1.to_v.weight], 0).detach()),
                w_o1=packing.pack_linear(blk.attn1.to_out[0].weight.detach()), b_o1=f32(blk.attn1.to_out[0].bias),
                w_q2=packing.pack_linear(blk.attn2.to_q.weight.detach()),
                w_kv2=packing.pack_linear(torch.cat([blk.attn2.to_k.weight, blk.attn2.to_v.weight], 0).detach()),
                w_o2=packing.pack_linear(blk.attn2.to_out[0].weight.detach()), b_o2=f32(blk.attn2.to_out[0].bias),
                w_ff1=wg, b_ff1=bg, ff_tile=tile,
                w_ff2=packing.pack_linear(blk.ff.net[2].weight.detach()), b_ff2=f32(blk.ff.net[2].bias))

        W["conv_in"] = dict(w=packing.pack_conv3x3_f32(self.conv_in.weight.detach()), b=f32(self.conv_in.bias))
        W["conv_out"] = dict(w=packing.pack_conv3x3_f32(self.conv_out.weight.detach()), b=f32(self.conv_out.bias),
                             g=f32(self.conv_norm_out.weight), beta=f32(self.conv_norm_out.bias),
                             w_tc=packing.pack_conv_out_tc(self.conv_out.weight.detach()))
        te = self.time_embedding
        W["temb"] = dict(w1=packing.pack_linear(te.linear_1.weight.detach()), b1=f32(te.linear_1.bias),
                         w2=packing.pack_linear(te.linear_2.weight.detach()), b2=f32(te.linear_2.bias))
        tp_w, tp_b = [], []
        for prefix, r in self._iter_resnets():
            res(prefix, r)
            tp_w.append(r.time_emb_proj.weight.detach())
            tp_b.append(r.time_emb_proj.bias.detach())
        W["tproj"] = dict(w=packing.pack_linear(torch.cat(tp_w, 0)), b=f32(torch.cat(tp_b, 0)))
        for prefix, a in self._iter_xformers():
            xf(prefix, a)
        for i, b in enumerate(self.down_blocks):
            if hasattr(b, "downsamplers"):
                W[f"down{i}.ds"] = dict(w=packing.pack_conv3x3(b.downsamplers[0].conv.weight.detach()),
                                        b=f32(b.downsamplers[0].conv.bias))
        for i, b in enumerate(self.up_blocks):
            if hasattr(b, "upsamplers"):
                W[f"up{i}.us"] = dict(w=packing.pack_conv3x3(b.upsamplers[0].conv.weight.detach()),
                                      b=f32(b.upsamplers[0].conv.bias))
        self._packed = W
        self._dirty = False
        self._param_versions = self._versions()

    def _ensure_packed(self):
        """(Re)pack the kernel-layout weights when the parameters changed; engines built on the old packing are dropped."""
        if self._dirty or self._packed is None or self._versions() != self._param_versions:
            self._pack_weights()
            self._engines = {}
            self.__dict__["_pack_gen"] = self.__dict__.get("_pack_gen", 0) + 1
        return self.__dict__.setdefault("_pack_gen", 0)

    def _stale(self, pack_gen):
        """True when plans built at packing generation `pack_gen` (CapturedSampler) no longer match the parameters."""
        return self._ensure_packed() != pack_gen

    def _versions(self):
        # called on EVERY forward: the parameter list is cached (walking the module tree costs ~1 ms for 686 parameters, which is
        # 20 % of a 5 ms denoising step on the host side); nn.Parameter objects are never replaced by .to() / load_state_dict()
        ps = self.__dict__.get("_param_list")
        if ps is None:
            ps = self.__dict__["_param_list"] = list(self.parameters())
        return sum([p._version for p in ps])

    def _iter_resnets(self):
        for i, b in enumerate(self.down_blocks):
            for j, r in enumerate(b.resnets):
                yield f"down{i}.res{j}", r
        for j, r in enumerate(self.mid_block.resnets):
            yield f"mid.res{j}", r
        for i, b in enumerate(self.up_blocks):
            for j, r in enumerate(b.resnets):
                yield f"up{i}.res{j}", r

    def _iter_xformers(self):
        for i, b in enumerate(self.down_blocks):
            if hasattr(b, "attentions"):
                for j, a in enumerate(b.attentions):
                    yield f"down{i}.attn{j}", a
        yield "mid.attn0", self.mid_block.attentions[0]
        for i, b in enumerate(self.up_blocks):
            if hasattr(b, "attentions"):
                for j, a in enumerate(b.attentions):
                    yield f"up{i}.attn{j}", a

    def _tproj_offsets(self):
        """All time_emb_proj heads run as ONE linear over their row-concatenation (in _iter_resnets order): ({resnet prefix:
        first output column of its head}, total columns)."""
        off, o = {}, 0
        for prefix, r in self._iter_resnets():
            off[prefix] = o
            o += r.cout
        return off, o

    def _walk(self, x, h, w, *, resnet, xformer, downsample, upsample, release):
        """Drive the down / mid / up blocks from conv_in's output x (h x w); returns (x, h, w) of the last up block.
            resnet(prefix, r, x, skip, h, w) -> y          skip: the down-path activation concatenated to x (None outside up)
            xformer(prefix, a, x, h, w) -> y
            downsample(prefix, s, x, h, w) -> y at h/2     s: the block's downsamplers[0]
            upsample(prefix, s, x, h, w) -> y at 2h        s: the block's upsamplers[0]
        The walk owns the skip stack and the liveness of activations: release(t) is called exactly once per activation, as
        soon as it is neither the running activation nor a pending skip (never for the returned one)."""
        skips = [x]

        def advance(y):         # y replaces x as the running activation
            nonlocal x
            if all(s is not x for s in skips):
                release(x)
            x = y

        for i, b in enumerate(self.down_blocks):
            for j, r in enumerate(b.resnets):
                advance(resnet(f"down{i}.res{j}", r, x, None, h, w))
                if hasattr(b, "attentions"):
                    advance(xformer(f"down{i}.attn{j}", b.attentions[j], x, h, w))
                skips.append(x)
            if hasattr(b, "downsamplers"):
                advance(downsample(f"down{i}.ds", b.downsamplers[0], x, h, w))
                h, w = h // 2, w // 2
                skips.append(x)
        mid = self.mid_block
        advance(resnet("mid.res0", mid.resnets[0], x, None, h, w))
        advance(xformer("mid.attn0", mid.attentions[0], x, h, w))
        advance(resnet("mid.res1", mid.resnets[1], x, None, h, w))
        for i, b in enumerate(self.up_blocks):
            for j, r in enumerate(b.resnets):
                skip = skips.pop()
                y = resnet(f"up{i}.res{j}", r, x, skip, h, w)
                if skip is not x and all(s is not skip for s in skips):
                    release(skip)
                advance(y)
                if hasattr(b, "attentions"):
                    advance(xformer(f"up{i}.attn{j}", b.attentions[j], x, h, w))
            if hasattr(b, "upsamplers"):
                advance(upsample(f"up{i}.us", b.upsamplers[0], x, h, w))
                h, w = 2 * h, 2 * w
        return x, h, w

    # -- forward --------------------------------------------------------------------------------
    def forward(self, sample, timestep, encoder_hidden_states, return_dict: bool = True):
        if sample.dim() != 4 or sample.shape[1] != self.in_channels:
            raise ValueError(f"sample must be (N, {self.in_channels}, H, W), got {tuple(sample.shape)}")
        ctx = encoder_hidden_states
        needs_grad = torch.is_grad_enabled() and (
            sample.requires_grad or ctx.requires_grad or any(p.requires_grad for p in self.parameters()) and self.training)
        if needs_grad and self.in_channels != 4:
            raise NotImplementedError(f"training a UNet with in_channels={self.in_channels} is not implemented (the inpainting "
                                      "UNet runs inference only): call it under torch.no_grad() or in eval mode")
        if not sample.is_cuda:
            raise B200SDError("b200sd.UNet2DConditionModel runs on CUDA only (no CPU fallback)")
        N, _, H, Wd = sample.shape
        n_down = len(self.config.block_out_channels) - 1
        if H % (1 << n_down) or Wd % (1 << n_down):
            raise ValueError(f"H and W must be multiples of {1 << n_down}")
        if ctx.dim() != 3 or ctx.shape[0] != N or ctx.shape[2] != self.config.cross_attention_dim:
            raise ValueError(f"encoder_hidden_states must be ({N}, S, {self.config.cross_attention_dim}), got {tuple(ctx.shape)}")
        if needs_grad:
            from .autograd import unet_forward_train
            out = unet_forward_train(self, sample, timestep, ctx)
            return UNet2DConditionOutput(sample=out) if return_dict else (out,)

        # version sum of the 686 parameters: catches in-place optimizer steps in eval mode too (the fused flat AdamW bumps no
        # version and calls mark_weights_changed() instead)
        self._ensure_packed()
        key = (N, H, Wd, ctx.shape[1], sample.device.index, self._precision)
        eng = self._engines.get(key)
        if eng is None:
            if self._precision == "fp32":
                from .engine_fp32 import EngineF32
                eng = EngineF32(self, N, H, Wd, ctx.shape[1], sample.device)
            else:
                from .engine import Engine
                eng = Engine(self, N, H, Wd, ctx.shape[1], sample.device)
            self._engines[key] = eng
        out = eng.run(sample, timestep, ctx, use_graph=self.use_cuda_graph)
        out = out.to(sample.dtype) if out.dtype != sample.dtype else out
        return UNet2DConditionOutput(sample=out) if return_dict else (out,)
