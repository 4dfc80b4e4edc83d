"""CLIP text encoder (SURVEY.md 8f N3): `transformers.CLIPTextModel`'s surface over b200sd kernels, forward AND backward.

Reference call sites: `CLIPTextModel.from_pretrained(path, subfolder="text_encoder")` finetune_sd.py:322-324;
`text_encoder = accelerator.prepare(text_encoder); text_encoder.train()` :375-379 (it is the TRAINED model of the reference's
default mode, `--train_text_encoder True` :29); `encoder_hidden_states = text_encoder(batch["input_ids"])[0]` :477;
`text_encoder.to(device, dtype=torch.float16)` + `freeze_params` :381-383 when the UNet trains instead.

Same module tree / state-dict keys as transformers (`text_model.embeddings.token_embedding.weight`,
`text_model.encoder.layers.{i}.self_attn.{q,k,v,out}_proj.{weight,bias}`, `...layer_norm{1,2}`, `...mlp.fc{1,2}`,
`text_model.final_layer_norm`), same `config.json` keys, `[0]` = last_hidden_state (B, 77, 768) fp32, `[1]` = pooled (EOS token).

Data flow per layer (tokens M = B * 77; each arrow = one kernel; the fp32 residual stream x is never rounded):
    x -LN1-> n1 -QKV GEMM(+bias)-> qkv -causal attention-> a -out GEMM(+bias +x)-> x1
    x1 -LN2-> n2 -fc1 GEMM(+bias)-> u -quick-GELU-> g -fc2 GEMM(+bias +x1)-> x'
The linears run on the tcgen05 GEMM (q|k|v fused into one [3C][C] matrix: the three weights are adjacent in the flat buffer),
their gradients on the dgrad / wgrad modes of the same kernel; embedding, causal attention, quick-GELU and the fp32-output
final LayerNorm are csrc/clip.cu.  State lives in train.FlatParams buffers (fp32 master = the parameters themselves, bf16
tensor-core copy, flat fp32 gradient) so that the data-parallel step allreduces ONE buffer and the fused AdamW kernel updates it.
There is no CPU / eager fallback.
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import ops
from ._lib import B200SDError
from .plan import Builder, Plan, capture, run_plan
from .train import F32, BF16, FlatParams

_CONFIG_DEFAULTS = dict(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12,
                        max_position_embeddings=77, layer_norm_eps=1e-5, hidden_act="quick_gelu", attention_dropout=0.0,
                        initializer_range=0.02, initializer_factor=1.0, pad_token_id=1, bos_token_id=49406, eos_token_id=49407,
                        projection_dim=768)


class CLIPTextConfig(SimpleNamespace):
    def __init__(self, **kw):
        super().__init__(**{**_CONFIG_DEFAULTS, **kw})

    def to_dict(self):
        return dict(vars(self))


class CLIPTextModelOutput(tuple):
    """(last_hidden_state, pooler_output) with attribute access, like transformers' BaseModelOutputWithPooling"""

    def __new__(cls, last_hidden_state, pooler_output):
        o = super().__new__(cls, (last_hidden_state, pooler_output))
        o.last_hidden_state, o.pooler_output = last_hidden_state, pooler_output
        return o


class _Attn(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.k_proj, self.v_proj, self.q_proj, self.out_proj = (nn.Linear(c, c) for _ in range(4))


class _MLP(nn.Module):
    def __init__(self, c, inter):
        super().__init__()
        self.fc1, self.fc2 = nn.Linear(c, inter), nn.Linear(inter, c)


class _Layer(nn.Module):
    def __init__(self, c, inter, eps):
        super().__init__()
        self.self_attn = _Attn(c)
        self.layer_norm1 = nn.LayerNorm(c, eps=eps)
        self.mlp = _MLP(c, inter)
        self.layer_norm2 = nn.LayerNorm(c, eps=eps)


class _Embeddings(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.token_embedding = nn.Embedding(cfg.vocab_size, cfg.hidden_size)
        self.position_embedding = nn.Embedding(cfg.max_position_embeddings, cfg.hidden_size)


class _Encoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.layers = nn.ModuleList(_Layer(cfg.hidden_size, cfg.intermediate_size, cfg.layer_norm_eps)
                                    for _ in range(cfg.num_hidden_layers))


class _TextTransformer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.embeddings = _Embeddings(cfg)
        self.encoder = _Encoder(cfg)
        self.final_layer_norm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)


class ClipFlat(FlatParams):
    """train.FlatParams for the text encoder: forward order, q|k|v weights (and biases) adjacent."""

    def _layout(self, m, add, add_adjacent):
        tm = m.text_model
        add(tm.embeddings.token_embedding.weight, "vec")
        add(tm.embeddings.position_embedding.weight, "vec")
        for L in tm.encoder.layers:
            add(L.layer_norm1.weight, "vec"); add(L.layer_norm1.bias, "vec")
            a = L.self_attn
            add_adjacent([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], "lin")
            add_adjacent([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias], "vec")
            add(a.out_proj.weight, "lin"); add(a.out_proj.bias, "vec")
            add(L.layer_norm2.weight, "vec"); add(L.layer_norm2.bias, "vec")
            add(L.mlp.fc1.weight, "lin"); add(L.mlp.fc1.bias, "vec")
            add(L.mlp.fc2.weight, "lin"); add(L.mlp.fc2.bias, "vec")
        add(tm.final_layer_norm.weight, "vec"); add(tm.final_layer_norm.bias, "vec")


class ClipEngine(Builder):
    """Forward launch plan (keeps what the backward needs: ~30 MB at 16 prompts) and backward launch plan for a fixed number
    of prompts; each is captured into a CUDA graph on first use."""

    def __init__(self, model, flat, B, S, device, train_weights):
        super().__init__(device)
        self.model, self.flat, self.B, self.S, self.train_weights = model, flat, B, S, train_weights
        self.fwd, self.bwd = Plan(), Plan()
        self.fwd_graph = self.bwd_graph = None
        self.use_graph = True
        self.forward_generation = 0
        with torch.cuda.device(device):
            self._build()

    # -- helpers (same contracts as train.TrainEngine's) ----------------------------------------------
    def P(self, p):
        r = self.flat.reg(p)
        return r.pview if r.pview.is_contiguous() else r.param.data

    def G(self, p):
        return self.flat.reg(p).g if self.train_weights else None

    def _new(self, rows, cols, dtype=BF16):
        return torch.empty(rows, cols, dtype=dtype, device=self.device)

    def _build(self):
        m, flat, B, S, dev = self.model, self.flat, self.B, self.S, self.device
        cfg = m.config
        C, I, heads = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads
        d = C // heads
        scale, eps = d ** -0.5, cfg.layer_norm_eps
        M = B * S
        tm = m.text_model
        Fp, Bp, tw = self.fwd, self.bwd, self.train_weights
        self.ids = torch.zeros(B, S, dtype=torch.int64, device=dev)
        self.out = torch.zeros(M, C, dtype=F32, device=dev)
        self.d_out = torch.zeros(M, C, dtype=F32, device=dev)
        tok, pos = tm.embeddings.token_embedding.weight, tm.embeddings.position_embedding.weight

        x = self._new(M, C, F32)
        Fp.append(lambda x=x: ops.clip_embed(self.ids, self.P(tok), self.P(pos), x))
        layers = []
        for L in tm.encoder.layers:
            a = L.self_attn
            w_qkv = flat.span([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], "wb")
            b_qkv = flat.span([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias], "master")
            wb = lambda p: flat.reg(p).wb
            n1, qkv, at = self._new(M, C), self._new(M, 3 * C), self._new(M, C)
            x1, n2, u, g, x2 = self._new(M, C, F32), self._new(M, C), self._new(M, I), self._new(M, I), self._new(M, C, F32)
            Fp.append(lambda x=x, L=L, n1=n1: ops.layernorm(x, self.P(L.layer_norm1.weight), self.P(L.layer_norm1.bias), n1, eps))
            self.gemm(Fp, n1, w_qkv, qkv, bias=b_qkv)
            Fp.append(lambda qkv=qkv, at=at: ops.causal_attention(qkv, at, B, heads, S, d, scale))
            self.gemm(Fp, at, wb(a.out_proj.weight), x1, bias=self.P(a.out_proj.bias), residual=x)
            Fp.append(lambda x1=x1, L=L, n2=n2: ops.layernorm(x1, self.P(L.layer_norm2.weight), self.P(L.layer_norm2.bias), n2, eps))
            self.gemm(Fp, n2, wb(L.mlp.fc1.weight), u, bias=self.P(L.mlp.fc1.bias))
            Fp.append(lambda u=u, g=g: ops.quick_gelu_fwd(u, g))
            self.gemm(Fp, g, wb(L.mlp.fc2.weight), x2, bias=self.P(L.mlp.fc2.bias), residual=x1)
            layers.append((L, x, n1, qkv, at, x1, n2, u, g, w_qkv))
            x = x2
        lnf = tm.final_layer_norm
        Fp.append(lambda x=x: ops.layernorm_f32out(x, self.P(lnf.weight), self.P(lnf.bias), self.out, eps))

        # ---- backward: dx is the fp32 gradient of the residual stream, updated in place from the last layer to the first ----
        dx = self._new(M, C, F32)
        d16 = self._new(M, C)
        dg, du, dn, da, dqkv = self._new(M, I), self._new(M, I), self._new(M, C), self._new(M, C), self._new(M, 3 * C)
        Bp.append(lambda: dx.zero_())
        Bp.append(lambda: ops.grad_prep(self.d_out, d16, None))
        Bp.append(lambda x=x: ops.layernorm_bwd(x, self.P(lnf.weight), d16, dx, self.G(lnf.weight), self.G(lnf.bias), eps))
        for (L, xin, n1, qkv, at, x1, n2, u, g, w_qkv) in reversed(layers):
            a = L.self_attn
            wb = lambda p: flat.reg(p).wb
            # x' = fc2(g) + x1
            Bp.append(lambda L=L: ops.grad_prep(dx, d16, self.G(L.mlp.fc2.bias)))
            self.wgrad(Bp, d16, g, self.G(L.mlp.fc2.weight))
            self.dgrad(Bp, d16, wb(L.mlp.fc2.weight), dg)
            Bp.append(lambda u=u: ops.quick_gelu_bwd(u, dg, du))
            if tw:
                Bp.append(lambda L=L: ops.grad_prep(du, None, self.G(L.mlp.fc1.bias)))
            self.wgrad(Bp, du, n2, self.G(L.mlp.fc1.weight))
            self.dgrad(Bp, du, wb(L.mlp.fc1.weight), dn)
            Bp.append(lambda x1=x1, L=L: ops.layernorm_bwd(x1, self.P(L.layer_norm2.weight), dn, dx, self.G(L.layer_norm2.weight),
                                                          self.G(L.layer_norm2.bias), eps))
            # x1 = out_proj(attention) + x
            Bp.append(lambda a=a: ops.grad_prep(dx, d16, self.G(a.out_proj.bias)))
            self.wgrad(Bp, d16, at, self.G(a.out_proj.weight))
            self.dgrad(Bp, d16, wb(a.out_proj.weight), da)
            Bp.append(lambda qkv=qkv: ops.causal_attention_bwd(qkv, da, dqkv, B, heads, S, d, scale))
            if tw:
                g_bqkv = flat.span([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias], "grad")
                Bp.append(lambda gb=g_bqkv: ops.grad_prep(dqkv, None, gb))
                self.wgrad(Bp, dqkv, n1, flat.span([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], "grad"))
            self.dgrad(Bp, dqkv, w_qkv, dn)
            Bp.append(lambda xin=xin, L=L: ops.layernorm_bwd(xin, self.P(L.layer_norm1.weight), dn, dx, self.G(L.layer_norm1.weight),
                                                            self.G(L.layer_norm1.bias), eps))
        if tw:
            Bp.append(lambda: ops.clip_embed_bwd(self.ids, dx, flat.reg(tok).gview, flat.reg(pos).gview))
        self.launches = (len(Fp), len(Bp))

    # -- execution ------------------------------------------------------------------------------------
    def _run(self, plan, which):
        g = getattr(self, which)
        if g is not None:
            g.replay()
        elif self.use_graph:
            setattr(self, which, capture(plan, "thread_local")[0])      # backward plans are captured on autograd's thread
        else:
            run_plan(plan)

    def run_forward(self, ids):
        with torch.cuda.device(self.device):
            self.flat.refresh_weights()
            self.ids.copy_(ids)
            self._run(self.fwd, "fwd_graph")
            self.forward_generation += 1
            return self.out

    def run_backward(self, d_out):
        with torch.cuda.device(self.device):
            self.d_out.copy_(d_out.reshape(self.d_out.shape))
            self._run(self.bwd, "bwd_graph")


class _ClipFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, ids, *params):
        ctx.engine, ctx.n_params = engine, len(params)
        ctx.param_ids = [id(p) for p in params]
        out = engine.run_forward(ids).clone()
        ctx.generation = engine.forward_generation
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_out):
        eng = ctx.engine
        if ctx.generation != eng.forward_generation:
            raise RuntimeError("b200sd: backward() of a text-encoder forward whose saved activations were overwritten by a later "
                               "forward of the same batch size: call backward() before the next training forward")
        model, flat = eng.model, eng.flat
        direct = model._direct_grads
        if not direct:
            flat.zero_grad()
        elif any(r.param.requires_grad and (r.param.grad is None or r.param.grad.data_ptr() != r.gview.data_ptr())
                 for r in flat.order):
            flat.zero_grad()
            flat.attach_grads()
        eng.run_backward(d_out.contiguous().float())
        if direct:
            return (None, None) + (None,) * ctx.n_params
        return (None, None) + tuple(flat.regs[i].gview if flat.regs[i].param.requires_grad else None for i in ctx.param_ids)


class CLIPTextModel(nn.Module):
    config_name = "config.json"

    def __init__(self, config=None, **kw):
        super().__init__()
        if config is None:
            config = CLIPTextConfig(**kw)
        elif isinstance(config, dict):
            config = CLIPTextConfig(**config)
        elif not isinstance(config, CLIPTextConfig):       # e.g. a transformers CLIPTextConfig
            config = CLIPTextConfig(**{k: getattr(config, k) for k in _CONFIG_DEFAULTS if hasattr(config, k)})
        if config.hidden_act != "quick_gelu":
            raise NotImplementedError("only hidden_act='quick_gelu' (SD v1.x text encoders) is implemented")
        if config.hidden_size % config.num_attention_heads or config.hidden_size % 64 or config.intermediate_size % 64:
            raise ValueError("hidden_size / intermediate_size must be multiples of 64, hidden_size divisible by the heads")
        self.config = config
        self.text_model = _TextTransformer(config)
        self._flat = None
        self._engines = {}
        self._direct_grads = False
        with torch.no_grad():                              # transformers' CLIPTextModel._init_weights
            f, c, n = config.initializer_factor, config.hidden_size, config.num_hidden_layers
            self.text_model.embeddings.token_embedding.weight.normal_(0.0, f * 0.02)
            self.text_model.embeddings.position_embedding.weight.normal_(0.0, f * 0.02)
            for L in self.text_model.encoder.layers:
                in_std, out_std, fc_std = c ** -0.5 * (2 * n) ** -0.5 * f, c ** -0.5 * f, (2 * c) ** -0.5 * f
                for lin, std in ((L.self_attn.q_proj, in_std), (L.self_attn.k_proj, in_std), (L.self_attn.v_proj, in_std),
                                 (L.self_attn.out_proj, out_std), (L.mlp.fc1, fc_std), (L.mlp.fc2, in_std)):
                    lin.weight.normal_(0.0, std)
                    lin.bias.zero_()

    # -- the surface the reference touches ------------------------------------------------------------
    @property
    def device(self):
        return self.text_model.final_layer_norm.weight.device

    @property
    def dtype(self):
        return self.text_model.final_layer_norm.weight.dtype

    def get_input_embeddings(self):
        return self.text_model.embeddings.token_embedding

    def gradient_checkpointing_enable(self, *a, **kw):
        """accepted for API compatibility (finetune_sd.py:378-379): the saved activations of the 12 layers are ~30 MB"""

    def enable_direct_gradients(self, enabled=True):
        """param.grad become views of ONE flat fp32 gradient buffer (what trainer.TextEncoderTrainer allreduces)"""
        self._direct_grads = bool(enabled)
        return self

    def flat_gradients(self):
        return None if self._flat is None else self._flat.grad

    def mark_weights_changed(self):
        """the engines read the flat buffers directly: nothing to repack (called by trainer.FlatAdamW)"""

    def zero_grad(self, set_to_none: bool = True):
        if self._direct_grads and self._flat is not None and self._flat.grad is not None:
            self._flat.zero_grad()
            self._flat.attach_grads()
            return
        super().zero_grad(set_to_none=set_to_none)

    def _apply(self, fn, *a, **kw):
        r = super()._apply(fn, *a, **kw)
        self._flat, self._engines = None, {}
        ps = list(self.parameters())
        if ps and all(p.is_cuda and p.dtype == torch.float32 and p.device == ps[0].device for p in ps):
            with torch.cuda.device(ps[0].device):          # re-home at .to(device) time: wrappers (DDP) must see final strides
                self._flat = ClipFlat(self, ps[0].device, lazy=True)
        return r

    def _ensure_flat(self, dev):
        if self._flat is None or self._flat.device != dev or not self._flat.owns(self):
            # fp16 / bf16 parameters (StableDiffusionPipeline.from_pretrained(torch_dtype=torch.float16), inference.py:406; the
            # frozen copy of finetune_sd.py:381) keep their own storage, the kernels read an fp32 upcast: inference only --
            # forward() refuses to TRAIN such a model
            self._flat = ClipFlat(self, dev, allow_half_trainable=True)
            self._engines = {}
        return self._flat.materialize()

    def forward(self, input_ids=None, attention_mask=None, position_ids=None, output_attentions=None, output_hidden_states=None,
                return_dict=None):
        if input_ids is None:
            raise ValueError("You have to specify input_ids")
        if attention_mask is not None or position_ids is not None or output_attentions or output_hidden_states:
            raise NotImplementedError("attention_mask / position_ids / output_* are not on the reference path (finetune_sd.py:477)")
        if not input_ids.is_cuda:
            raise B200SDError("b200sd.CLIPTextModel runs on CUDA only (no CPU fallback)")
        cfg = self.config
        ids = input_ids.reshape(-1, input_ids.shape[-1])
        B, S = ids.shape
        if S > cfg.max_position_embeddings:
            raise ValueError(f"sequence length {S} exceeds max_position_embeddings {cfg.max_position_embeddings}")
        dev = ids.device
        flat = self._ensure_flat(dev)
        train = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if train and self.dtype != torch.float32:
            raise B200SDError("training the text encoder needs fp32 master parameters (the kernels compute in bf16 on their own "
                              "copy); run a half-precision model under torch.no_grad() or freeze it (requires_grad_(False))")
        key = (B, S, dev.index, train)
        eng = self._engines.get(key)
        if eng is None:
            eng = self._engines[key] = ClipEngine(self, flat, B, S, dev, train_weights=train)
        if train:
            out = _ClipFn.apply(eng, ids, *list(self.parameters()))
        else:
            out = eng.run_forward(ids).clone()
        last = out.view(B, S, cfg.hidden_size)
        if self.dtype != torch.float32:
            last = last.to(self.dtype)
        # pooled output = hidden state at the EOS token (argmax of the ids in transformers 4.29.2: EOS is the largest id)
        pooled = last[torch.arange(B, device=dev), ids.argmax(dim=-1)]
        return CLIPTextModelOutput(last, pooled)

    # -- (de)serialisation in the transformers directory layout ---------------------------------------
    @classmethod
    def from_pretrained(cls, path, subfolder=None, torch_dtype=None, **kw):
        d = path if subfolder is None else os.path.join(path, subfolder)
        with open(os.path.join(d, cls.config_name)) as f:
            cfg = json.load(f)
        model = cls(**{k: v for k, v in cfg.items() if k in _CONFIG_DEFAULTS})
        st_path, bin_path = os.path.join(d, "model.safetensors"), os.path.join(d, "pytorch_model.bin")
        if os.path.exists(st_path):
            from safetensors.torch import load_file
            sd = load_file(st_path)
        elif os.path.exists(bin_path):
            sd = torch.load(bin_path, map_location="cpu")
        else:
            raise FileNotFoundError(f"no model.safetensors / pytorch_model.bin under {d}")
        sd = {k: v for k, v in sd.items() if not k.endswith("position_ids")}      # a buffer in transformers < 4.31 checkpoints
        model.load_state_dict(sd, strict=True)
        if torch_dtype is not None:
            model.to(dtype=torch_dtype)
        return model.eval()

    def save_pretrained(self, path, safe_serialization=False):
        os.makedirs(path, exist_ok=True)
        cfg = dict(self.config.to_dict(), architectures=["CLIPTextModel"], model_type="clip_text_model")
        with open(os.path.join(path, self.config_name), "w") as f:
            json.dump(cfg, f, indent=2)
        sd = {k: v.detach().cpu().contiguous() for k, v in self.state_dict().items()}
        if safe_serialization:
            from safetensors.torch import save_file
            save_file(sd, os.path.join(path, "model.safetensors"))
        else:
            torch.save(sd, os.path.join(path, "pytorch_model.bin"))
