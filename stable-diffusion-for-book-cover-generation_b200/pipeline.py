"""The denoising loop of StableDiffusionPipeline.__call__ (SURVEY.md App. B.4) -- the part of the
pipeline that is on the hot path.  Tokeniser / CLIP / VAE stay outside (neighbours, out of scope):
callers pass the (2B, 77, 768) context `cat([uncond, cond])` and the initial latents.

Reference call sites: inference.py:175-176, 342-351; finetune_sd.py:264-271."""
from __future__ import annotations

import inspect

import torch

from . import ops
from .schedulers import SCHEDULERS


@torch.no_grad()
def denoise_loop(unet, scheduler, latents, encoder_hidden_states_2b, num_inference_steps=50, guidance_scale=7.5,
                 record=None, eta=0.0, generator=None, start=0, blend=None, cond=None):
    """latents (B,4,h,w) -> denoised latents (B,4,h,w).  One UNet call at batch 2B per step, then ONE
    fused kernel for `eps_u + s (eps_c - eps_u)` + the scheduler update.  As in diffusers, `eta` and `generator` reach only
    a scheduler whose step takes them (eta: DDIM; generator: DDIM and DDPM).

    img2img / legacy inpainting: the loop runs over timesteps[start:] (no step when that is empty).  blend=(init_orig, noise,
    mask) adds legacy inpainting's masking step after every scheduler step at loop timestep t:
    latents = mask * add_noise(init_orig, noise, t) + (1 - mask) * latents, mask broadcastable to the latents (1 = keep).

    9-channel inpainting UNet: cond = cat([mask, masked_image_latents], 1) (B, 5, h, w) joins every step's UNet input in
    diffusers 0.7.2's order -- cat([latents] * 2), cat with cat([cond] * 2) along the channels, then scale_model_input."""
    if encoder_hidden_states_2b.shape[0] != 2 * latents.shape[0]:
        raise ValueError("encoder_hidden_states must be cat([uncond, cond]) with batch 2B")
    in_channels = getattr(getattr(unet, "config", None), "in_channels", latents.shape[1])
    n_cond = in_channels - latents.shape[1]
    if (cond is None) != (n_cond == 0) or (cond is not None and tuple(cond.shape) != (latents.shape[0], n_cond) + tuple(latents.shape[2:])):
        raise ValueError(f"a UNet with in_channels={in_channels} takes {latents.shape[1]}-channel latents and "
                         + (f"cond (B, {n_cond}, h, w) = [mask | masked-image latents], got "
                            f"{None if cond is None else tuple(cond.shape)}" if n_cond else "no cond"))
    if cond is not None and (start != 0 or blend is not None):
        raise ValueError("the 9-channel inpainting UNet runs the full schedule from noise: no start step and no blend")
    scheduler.set_timesteps(num_inference_steps)
    timesteps = scheduler.timesteps.tolist()[start:]
    accepted = inspect.signature(scheduler.step_cfg).parameters
    extra = {k: v for k, v in (("eta", eta), ("generator", generator)) if k in accepted}
    sampler = (_captured_sampler(unet, scheduler, latents, encoder_hidden_states_2b, guidance_scale, extra.get("eta", 0.0),
                                 start, blend is not None)
               if record is None and timesteps else None)
    if sampler is not None:
        cond_args = None if cond is None else (cond[:, :1], cond[:, 1:])
        return sampler.run(latents, encoder_hidden_states_2b, generator, blend=blend, cond=cond_args).to(latents.dtype)
    latents = (latents * scheduler.init_noise_sigma).float().contiguous()
    if blend is not None:
        init_orig, noise, mask = (t.to(latents.device).float() for t in blend)
        init_orig, noise, mask = init_orig.contiguous(), noise.contiguous(), mask.expand_as(latents).contiguous()
        tables = scheduler._noise_tables(latents.device)
    x2 = torch.empty((2 * latents.shape[0],) + tuple(latents.shape[1:]), dtype=latents.dtype, device=latents.device)
    B = latents.shape[0]
    cond2 = None if cond is None else torch.cat([cond.to(latents.device, latents.dtype)] * 2)
    for t in timesteps:
        x2[:B].copy_(latents)
        x2[B:].copy_(latents)
        x_in = x2 if cond2 is None else torch.cat([x2, cond2], dim=1)
        eps2 = unet(scheduler.scale_model_input(x_in, t), t, encoder_hidden_states_2b).sample
        if record is not None:
            record.append(eps2[:B] + guidance_scale * (eps2[B:] - eps2[:B]))
        latents = scheduler.step_cfg(eps2.float() if eps2.dtype not in (torch.float32, torch.bfloat16) else eps2, t,
                                     latents, guidance_scale, **extra).prev_sample
        if blend is not None:
            latents = ops.inpaint_blend(latents.contiguous(), init_orig, noise, mask, t, *tables)
    return latents


def _captured_sampler(unet, scheduler, latents, ctx2, guidance_scale, eta=0.0, start=0, inpaint=False):
    """The whole-step CUDA graph (sampler.CapturedSampler) when the combination is covered: b200sd UNet on its bf16 plan with
    CUDA graphs on, DDIM, PLMS, DDPM, LMS, Euler or Euler-ancestral, CUDA tensors.  Cached on the UNet per (geometry, schedule,
    guidance, eta, start step, inpaint mode); None -> the per-call loop."""
    from .unet import UNet2DConditionModel
    if not (isinstance(unet, UNet2DConditionModel) and hasattr(scheduler, "captured_step") and latents.is_cuda
            and unet._precision == "bf16" and unet.use_cuda_graph and not unet.training):
        return None
    from .sampler import CapturedSampler
    B, _, h, w = latents.shape
    key = (type(scheduler).__name__, B, h, w, ctx2.shape[1], latents.device.index, float(guidance_scale), float(eta),
           tuple(scheduler.timesteps.tolist()), tuple(sorted((k, str(v)) for k, v in vars(scheduler.config).items())),
           int(start), bool(inpaint))
    cache = unet.__dict__.setdefault("_samplers", {})
    smp = cache.get(key)
    if smp is not None and unet._stale(smp._pack_gen):
        cache.clear()
        smp = None
    if smp is None:
        if len(cache) >= 4:
            cache.clear()          # each sampler owns a full set of activation buffers
        smp = cache[key] = CapturedSampler(unet, scheduler, B, h, w, ctx2.shape[1], guidance_scale, eta=eta, start=start,
                                           inpaint=inpaint)
    return smp


# ---------------------------------------------------------------------------------------------------
# StableDiffusionPipeline-compatible wrapper (SURVEY.md 8f N4): what finetune_sd.py:517-537 builds and saves,
# what utils.py:181-256 / inference.py:404-429 load, and what inference.py:175-176, 342-351 call.
# UNet, scheduler, text encoder (clip.py) and VAE (vae.py) are b200sd's; objects the caller passes instead (transformers'
# CLIPTextModel, a diffusers AutoencoderKL) are used as they are.  The tokenizer is transformers' CLIPTokenizer (host code).
# ---------------------------------------------------------------------------------------------------
import json
import os
from types import SimpleNamespace

_SCHEDULERS = tuple(cls.__name__ for cls in SCHEDULERS)


class StableDiffusionPipelineOutput(SimpleNamespace):
    """`.images` (list of PIL images, or a tensor for output_type "pt" / "latent") and `.nsfw_content_detected` (None)."""


_INPAINT_CHANNELS = 4 + 1 + 4      # latents | mask | masked-image latents: the UNet of diffusers' StableDiffusionInpaintPipeline


def _latent_channels(unet):
    """the channel count of the latents `unet` denoises; a 9-channel inpainting UNet has no place in the 4-channel pipelines"""
    if unet.in_channels == _INPAINT_CHANNELS:
        raise ValueError(f"this UNet has in_channels={_INPAINT_CHANNELS} (an inpainting UNet): use StableDiffusionInpaintPipeline")
    return unet.in_channels


class StableDiffusionPipeline:
    """Same constructor keywords, `save_pretrained` / `from_pretrained` directory layout (`model_index.json` + one sub-folder
    per component) and `__call__` signature as diffusers 0.7.2's pipeline.  `safety_checker` / `feature_extractor` are
    accepted and ignored (the reference always passes `safety_checker=None`: inference.py:407, 427; utils.py:190, 225, 250)."""

    config_name = "model_index.json"
    _saved_class_name = "StableDiffusionPipeline"     # model_index.json's _class_name

    def __init__(self, vae=None, text_encoder=None, tokenizer=None, unet=None, scheduler=None, safety_checker=None,
                 feature_extractor=None):
        if unet is None or scheduler is None:
            raise ValueError("StableDiffusionPipeline needs at least `unet` and `scheduler`")
        self.vae, self.text_encoder, self.tokenizer = vae, text_encoder, tokenizer
        self.unet, self.scheduler = unet, scheduler
        self.safety_checker, self.feature_extractor = None, feature_extractor
        self._progress_bar_config = {}

    # -- housekeeping the reference touches ----------------------------------------------------------
    @property
    def device(self):
        return self.unet.device

    def to(self, device=None, dtype=None):
        for name in ("unet", "text_encoder", "vae"):
            m = getattr(self, name)
            if m is not None and hasattr(m, "to"):
                setattr(self, name, m.to(device) if dtype is None else m.to(device, dtype=dtype))
        return self

    def set_progress_bar_config(self, **kw):
        self._progress_bar_config = kw

    def enable_attention_slicing(self, *a, **kw):
        """accepted no-op: the fused attention kernel never materialises the S x S scores that slicing exists to bound"""

    disable_attention_slicing = enable_attention_slicing

    @property
    def components(self):
        return dict(vae=self.vae, text_encoder=self.text_encoder, tokenizer=self.tokenizer, unet=self.unet,
                    scheduler=self.scheduler, safety_checker=None, feature_extractor=self.feature_extractor)

    # -- (de)serialisation in the diffusers directory layout -----------------------------------------
    def save_pretrained(self, path, safe_serialization=False):
        os.makedirs(path, exist_ok=True)
        index = {"_class_name": self._saved_class_name, "_diffusers_version": "0.7.2"}
        for name, obj in self.components.items():
            if obj is None:
                index[name] = [None, None]
                continue
            lib = "diffusers" if name in ("unet", "scheduler", "vae") else "transformers"
            index[name] = [lib, type(obj).__name__]
            sub = os.path.join(path, name)
            if name == "unet":
                obj.save_pretrained(sub, safe_serialization=safe_serialization)
            elif hasattr(obj, "save_pretrained"):
                obj.save_pretrained(sub)
        with open(os.path.join(path, self.config_name), "w") as f:
            json.dump(index, f, indent=2)

    @classmethod
    def from_pretrained(cls, path, torch_dtype=None, safety_checker=None, scheduler=None, **overrides):
        """Loads `unet/` and `scheduler/` with b200sd's classes, and the text encoder / VAE with b200sd's when their
        `text_encoder/` and `vae/` sub-folders exist (b200sd.clip.CLIPTextModel, b200sd.vae.AutoencoderKL); the tokenizer through
        transformers (offline)."""
        from . import schedulers as S
        from .unet import UNet2DConditionModel
        with open(os.path.join(path, cls.config_name)) as f:
            index = json.load(f)
        unet = overrides.pop("unet", None) or UNet2DConditionModel.from_pretrained(path, subfolder="unet", torch_dtype=torch_dtype)
        if scheduler is None:
            cls_name = (index.get("scheduler") or [None, "PNDMScheduler"])[1]
            with open(os.path.join(path, "scheduler", "scheduler_config.json")) as f:
                cls_name = json.load(f).get("_class_name", cls_name)
            if cls_name not in _SCHEDULERS:
                raise ValueError(f"scheduler class {cls_name!r} is not implemented ({', '.join(_SCHEDULERS)} are)")
            kw = {"skip_prk_steps": True} if cls_name == "PNDMScheduler" else {}
            scheduler = getattr(S, cls_name).from_config(path, subfolder="scheduler", **kw)
        tokenizer, text_encoder = overrides.pop("tokenizer", None), overrides.pop("text_encoder", None)
        if tokenizer is None and os.path.isdir(os.path.join(path, "tokenizer")):
            from transformers import CLIPTokenizer
            tokenizer = CLIPTokenizer.from_pretrained(os.path.join(path, "tokenizer"))
        if text_encoder is None and os.path.isdir(os.path.join(path, "text_encoder")):
            from .clip import CLIPTextModel
            text_encoder = CLIPTextModel.from_pretrained(path, subfolder="text_encoder", torch_dtype=torch_dtype)
        vae = overrides.pop("vae", None)
        if vae is None and os.path.isdir(os.path.join(path, "vae")):
            from .vae import AutoencoderKL
            vae = AutoencoderKL.from_pretrained(path, subfolder="vae", torch_dtype=torch_dtype)
        return cls(vae=vae, text_encoder=text_encoder, tokenizer=tokenizer, unet=unet,
                   scheduler=scheduler, safety_checker=None, feature_extractor=overrides.pop("feature_extractor", None))

    # -- sampling ------------------------------------------------------------------------------------
    def _encode_prompt(self, prompt, negative_prompt, device):
        if self.tokenizer is None or self.text_encoder is None:
            raise ValueError("prompt strings need a tokenizer and a text_encoder; pass `prompt_embeds` (2B, 77, 768) instead")
        tok = lambda texts: self.tokenizer(texts, padding="max_length", max_length=self.tokenizer.model_max_length,
                                           truncation=True, return_tensors="pt").input_ids.to(device)
        cond = self.text_encoder(tok(prompt))[0]
        uncond = self.text_encoder(tok(negative_prompt if negative_prompt is not None else [""] * len(prompt)))[0]
        return torch.cat([uncond, cond])          # App. B.4: row block 0 = unconditional

    def _context(self, prompt, negative_prompt, prompt_embeds):
        """cat([uncond, cond]) (2B, 77, 768) on the pipeline's device, from prompt strings or as given"""
        if prompt_embeds is not None:
            return prompt_embeds.to(self.device)
        prompt = [prompt] if isinstance(prompt, str) else list(prompt)
        return self._encode_prompt(prompt, [negative_prompt] * len(prompt) if isinstance(negative_prompt, str) else negative_prompt,
                                   self.device)

    def _output(self, lat, output_type, return_dict):
        """decode -> `output_type` ("pil", "pt"; "latent" or no VAE: the latents) -> StableDiffusionPipelineOutput"""
        if output_type == "latent" or self.vae is None:
            images = lat
        else:
            dec = self.vae.decode(lat.to(next(self.vae.parameters()).dtype) / 0.18215)
            img = (getattr(dec, "sample", dec) / 2 + 0.5).clamp(0, 1)
            if output_type == "pt":
                images = img
            else:
                arr = (img.permute(0, 2, 3, 1).float().cpu().numpy() * 255).round().astype("uint8")
                from PIL import Image
                images = [Image.fromarray(a) for a in arr]
        out = StableDiffusionPipelineOutput(images=images, nsfw_content_detected=None)
        return out if return_dict else (images, None)

    @torch.no_grad()
    def __call__(self, prompt=None, height=512, width=512, num_inference_steps=50, guidance_scale=7.5, negative_prompt=None,
                 eta=0.0, generator=None, latents=None, output_type="pil", return_dict=True, prompt_embeds=None, **kw):
        """inference.py:175-176, 342-351: `pipeline(prompts, height=, width=, num_inference_steps=50, guidance_scale=7.5,
        latents=...)`.  `prompt_embeds` = cat([uncond, cond]) lets a caller without CLIP drive the hot path directly.
        `generator` draws the initial latents, then the step noise of DDPM / DDIM with eta > 0; `eta` reaches DDIM only."""
        if height % 8 or width % 8:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        device = self.device
        ctx2 = self._context(prompt, negative_prompt, prompt_embeds)
        B = ctx2.shape[0] // 2
        shape = (B, _latent_channels(self.unet), height // 8, width // 8)
        if latents is None:
            latents = _randn(shape, generator, device)
        elif tuple(latents.shape) != shape:
            raise ValueError(f"Unexpected latents shape, got {tuple(latents.shape)}, expected {shape}")
        lat = denoise_loop(self.unet, self.scheduler, latents.to(device).float(), ctx2.float(), num_inference_steps, guidance_scale,
                           eta=eta, generator=generator)
        return self._output(lat, output_type, return_dict)


def _randn(shape, generator, device):
    """torch.randn on the generator's device (the pipeline's when there is none), moved to the pipeline's device"""
    return torch.randn(shape, generator=generator, device=device if generator is None or generator.device.type != "cpu"
                       else "cpu").to(device)


# ---------------------------------------------------------------------------------------------------
# diffusers 0.7.2's StableDiffusionImg2ImgPipeline and StableDiffusionInpaintPipelineLegacy: they load the directory the
# training script saves (a StableDiffusionPipeline) and start the denoising loop partway through the schedule, from the
# noised latents of an init image.  Semantics as in 0.7.2, quirks kept: the entry point into the schedule
# (`scheduler.img2img_start`) and the masking step that re-noises the kept region with the current loop timestep.
# ---------------------------------------------------------------------------------------------------
def preprocess_image(image):
    """PIL image -> (1, 3, H, W) in [-1, 1]: width and height rounded down to multiples of 32, LANCZOS resize"""
    import numpy as np
    from PIL import Image
    image = image.convert("RGB")
    w, h = (v - v % 32 for v in image.size)
    arr = np.array(image.resize((w, h), resample=Image.LANCZOS)).astype(np.float32) / 255.0
    return 2.0 * torch.from_numpy(arr[None].transpose(0, 3, 1, 2).copy()) - 1.0


def preprocess_mask(mask):
    """PIL mask -> (1, 4, h/8, w/8) keep-mask: "L", rounded down to multiples of 32, NEAREST resize to latent size, /255,
    tiled to 4 channels, inverted (white = repaint, so 1 = keep).  Not binarised."""
    import numpy as np
    from PIL import Image
    mask = mask.convert("L")
    w, h = (v - v % 32 for v in mask.size)
    arr = np.array(mask.resize((w // 8, h // 8), resample=Image.NEAREST)).astype(np.float32) / 255.0
    return 1 - torch.from_numpy(np.tile(arr, (4, 1, 1))[None].copy())


class StableDiffusionImg2ImgPipeline(StableDiffusionPipeline):
    """diffusers 0.7.2's image-to-image pipeline: `pipe(prompt, init_image=, strength=0.8, ...)`.  init_image is a PIL image or a
    (B, 3, H, W) tensor in [-1, 1] (H, W multiples of 8) whose batch is 1 or the prompt count.  strength in [0, 1]: how far
    into the schedule the init latents are noised, i.e. how much of the image is repainted."""

    @torch.no_grad()
    def __call__(self, prompt=None, init_image=None, strength=0.8, num_inference_steps=50, guidance_scale=7.5,
                 negative_prompt=None, eta=0.0, generator=None, output_type="pil", return_dict=True, prompt_embeds=None):
        return self._from_image(prompt, init_image, None, strength, num_inference_steps, guidance_scale, negative_prompt, eta,
                                generator, output_type, return_dict, prompt_embeds)

    def _from_image(self, prompt, init_image, mask_image, strength, num_inference_steps, guidance_scale, negative_prompt, eta,
                    generator, output_type, return_dict, prompt_embeds):
        t_start, t_noise = self.scheduler.img2img_start(num_inference_steps, strength)     # checks strength first
        if init_image is None or self.vae is None:
            raise ValueError("image-to-image needs an init_image and a vae")
        device = self.device
        image = init_image if isinstance(init_image, torch.Tensor) else preprocess_image(init_image)
        if image.dim() != 4 or image.shape[1] != 3 or image.shape[2] % 8 or image.shape[3] % 8:
            raise ValueError(f"init_image must be (B, 3, H, W) with H and W multiples of 8, got {tuple(image.shape)}")
        ctx2 = self._context(prompt, negative_prompt, prompt_embeds)
        B = ctx2.shape[0] // 2
        if image.shape[0] not in (1, B):
            raise ValueError(f"init_image has batch {image.shape[0]}; it must be 1 or the prompt count {B}")
        shape = (B, _latent_channels(self.unet), image.shape[2] // 8, image.shape[3] // 8)
        mask = None
        if mask_image is not None:
            mask = mask_image if isinstance(mask_image, torch.Tensor) else preprocess_mask(mask_image)
            if mask.dim() != 4 or mask.shape[0] not in (1, B) or tuple(mask.shape[1:]) != shape[1:]:
                raise ValueError(f"The mask and init_image should be the same size: mask {tuple(mask.shape)}, init latents {shape}")
            mask = mask.to(device).float().expand(shape)
        vae_dtype = next(self.vae.parameters()).dtype
        init = 0.18215 * self.vae.encode(image.to(device, vae_dtype)).latent_dist.sample(generator).float()
        init = init.expand(shape) if init.shape[0] == 1 else init
        noise = _randn(shape, generator, device)
        latents = self.scheduler.add_noise(init.contiguous(), noise, torch.tensor([t_noise] * B))
        blend = None if mask is None else (init, noise, mask)
        lat = denoise_loop(self.unet, self.scheduler, latents, ctx2.float(), num_inference_steps, guidance_scale, eta=eta,
                           generator=generator, start=t_start, blend=blend)
        return self._output(lat, output_type, return_dict)


class StableDiffusionInpaintPipelineLegacy(StableDiffusionImg2ImgPipeline):
    """diffusers 0.7.2's legacy inpainting pipeline on the ordinary 4-channel UNet: img2img that keeps the region outside the
    mask.  mask_image: a PIL image (white = repaint) or a (1 or B, 4, h, w) keep-mask tensor at latent resolution (1 = keep).
    After every scheduler step at loop timestep t, latents = mask * add_noise(init, noise, t) + (1 - mask) * latents."""

    @torch.no_grad()
    def __call__(self, prompt=None, init_image=None, mask_image=None, strength=0.8, num_inference_steps=50, guidance_scale=7.5,
                 negative_prompt=None, eta=0.0, generator=None, output_type="pil", return_dict=True, prompt_embeds=None):
        if mask_image is None:
            raise ValueError("mask_image is required")
        return self._from_image(prompt, init_image, mask_image, strength, num_inference_steps, guidance_scale, negative_prompt,
                                eta, generator, output_type, return_dict, prompt_embeds)


# ---------------------------------------------------------------------------------------------------
# diffusers 0.7.2's StableDiffusionInpaintPipeline: the dedicated inpainting checkpoint, a UNet with in_channels = 9 that sees
# the mask and the masked image's latents at every step.  It starts from pure noise over the full schedule (no strength).
# ---------------------------------------------------------------------------------------------------
def prepare_mask_and_masked_image(image, mask):
    """0.7.2's prepare_mask_and_masked_image -> (mask (1|B, 1, H, W) in {0, 1}, masked image (1|B, 3, H, W) in [-1, 1]).
    PIL image: "RGB", NCHW, / 127.5 - 1, not resized.  PIL mask: "L", / 255.  Tensors: an image in [-1, 1] and a mask in [0, 1].
    The mask is binarised (< 0.5 -> 0, >= 0.5 -> 1; white = 1 = repaint) and the masked image keeps the pixels where it is 0."""
    import numpy as np
    if isinstance(image, torch.Tensor):
        image = image.float()
    else:
        arr = np.array(image.convert("RGB"))[None].transpose(0, 3, 1, 2)
        image = torch.from_numpy(arr.copy()).to(dtype=torch.float32) / 127.5 - 1.0
    if isinstance(mask, torch.Tensor):
        mask = mask.float()
    else:
        mask = torch.from_numpy((np.array(mask.convert("L")).astype(np.float32) / 255.0)[None, None].copy())
    if image.dim() != 4 or mask.dim() != 4 or image.shape[2:] != mask.shape[2:]:
        raise ValueError(f"image (B, 3, H, W) and mask_image (B, 1, H, W) must have the same height and width, got "
                         f"{tuple(image.shape)} and {tuple(mask.shape)}")
    mask = torch.where(mask < 0.5, torch.zeros_like(mask), torch.ones_like(mask))
    masked_image = image * (mask.to(image.device) < 0.5)
    return mask, masked_image


def latent_mask(mask, h, w):
    """the inpainting mask at latent size h x w: F.interpolate's default mode (nearest), as 0.7.2 resizes it"""
    import torch.nn.functional as F
    return F.interpolate(mask, size=(h, w))


class StableDiffusionInpaintPipeline(StableDiffusionPipeline):
    """diffusers 0.7.2's inpainting pipeline on a UNet with in_channels = 9: `pipe(prompt, image=, mask_image=, height=512,
    width=512, ...)`.  image: a PIL image or a (1 or B, 3, H, W) tensor in [-1, 1]; mask_image: a PIL image or a (1 or B, 1, H,
    W) tensor in [0, 1], white (>= 0.5) = repaint.  Both must already be height x width.  Every step's UNet input is
    [latents | mask | masked-image latents], the mask nearest-resized to the latents; the run draws from `generator` the initial
    latents, then the masked image's posterior sample, then the step noise."""

    _saved_class_name = "StableDiffusionInpaintPipeline"

    @torch.no_grad()
    def __call__(self, prompt=None, image=None, mask_image=None, height=512, width=512, num_inference_steps=50,
                 guidance_scale=7.5, negative_prompt=None, eta=0.0, generator=None, latents=None, output_type="pil",
                 return_dict=True, prompt_embeds=None):
        if height % 8 or width % 8:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if self.unet.in_channels != _INPAINT_CHANNELS:
            raise ValueError(f"Incorrect configuration settings! The config of `pipeline.unet` expects "
                             f"{self.unet.in_channels} input channels, but 4 (latents) + 1 (mask) + 4 (masked image latents) "
                             f"= {_INPAINT_CHANNELS} are passed: StableDiffusionInpaintPipeline needs the 9-channel inpainting UNet")
        if image is None or mask_image is None or self.vae is None:
            raise ValueError("inpainting needs an image, a mask_image and a vae")
        mask, masked_image = prepare_mask_and_masked_image(image, mask_image)
        if masked_image.dim() != 4 or masked_image.shape[1] != 3 or tuple(masked_image.shape[2:]) != (height, width):
            raise ValueError(f"image must be (B, 3, {height}, {width}) (height x width; it is not resized), got "
                             f"{tuple(masked_image.shape)}")
        if mask.dim() != 4 or mask.shape[1] != 1 or tuple(mask.shape[2:]) != (height, width):
            raise ValueError(f"mask_image must be (B, 1, {height}, {width}) (height x width; it is not resized), got {tuple(mask.shape)}")
        device = self.device
        ctx2 = self._context(prompt, negative_prompt, prompt_embeds)
        B = ctx2.shape[0] // 2
        for name, t in (("image", image), ("mask_image", mask)):
            if isinstance(t, torch.Tensor) and t.shape[0] not in (1, B):
                raise ValueError(f"{name} has batch {t.shape[0]}; it must be 1 or the prompt count {B}")
        shape = (B, self.unet.config.out_channels, height // 8, width // 8)
        if latents is None:
            latents = _randn(shape, generator, device)                      # first draw: the initial latents
        elif tuple(latents.shape) != shape:
            raise ValueError(f"Unexpected latents shape, got {tuple(latents.shape)}, expected {shape}")
        mask = latent_mask(mask, *shape[2:])
        vae_dtype = next(self.vae.parameters()).dtype
        masked_latents = 0.18215 * self.vae.encode(masked_image.to(device, vae_dtype)).latent_dist.sample(generator).float()
        cond = torch.cat([mask.to(device).expand(B, -1, -1, -1), masked_latents.expand(B, -1, -1, -1)], dim=1).contiguous()
        lat = denoise_loop(self.unet, self.scheduler, latents.to(device).float(), ctx2.float(), num_inference_steps, guidance_scale,
                           eta=eta, generator=generator, cond=cond)
        return self._output(lat, output_type, return_dict)
