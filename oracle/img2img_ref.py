"""ORACLE (test infrastructure, not product code) -- diffusers 0.7.2's StableDiffusionImg2ImgPipeline and
StableDiffusionInpaintPipelineLegacy restated in plain fp32 PyTorch + numpy, on the oracle UNet, VAE and schedulers
(oracle.unet_ref, oracle.vae_ref, oracle.schedulers_ref, oracle.ancestral_ref).  The quirks of 0.7.2 are kept: the noised init
latents sit at timesteps[-init_timestep] (timesteps[0] when init_timestep is 0), PLMS's call counter starts at 0 on the first
executed timestep, and the masking step re-noises the kept region at the current loop timestep with the same init noise.

Every random draw is an explicit argument (the posterior noise, the init noise; the step noise comes from `generator` as in
ancestral_ref), so tests can feed the product and the oracle identical draws.  No published known answer of these pipelines
exists in the tree, so none is claimed.
"""
from __future__ import annotations

import inspect

import numpy as np
import torch

from . import schedulers_ref as R


def preprocess_image(image):
    """PIL -> (1, 3, H, W) in [-1, 1]: sizes rounded down to multiples of 32, LANCZOS, /255, NCHW, 2x - 1"""
    from PIL import Image
    w, h = image.size
    w, h = w - w % 32, h - h % 32
    arr = np.array(image.resize((w, h), resample=Image.LANCZOS)).astype(np.float32) / 255.0
    return 2.0 * torch.from_numpy(arr[None].transpose(0, 3, 1, 2).copy()) - 1.0


def preprocess_mask(mask):
    """PIL -> (1, 4, h/8, w/8): "L", rounded down to multiples of 32, NEAREST to latent size, /255, 4 channels, 1 - mask"""
    from PIL import Image
    mask = mask.convert("L")
    w, h = mask.size
    w, h = w - w % 32, h - h % 32
    arr = np.array(mask.resize((w // 8, h // 8), resample=Image.NEAREST)).astype(np.float32) / 255.0
    arr = np.tile(arr, (4, 1, 1))[None]
    return torch.from_numpy(1 - arr)


def img2img_start(scheduler, num_inference_steps, strength):
    """(t_start, t_noise) after scheduler.set_timesteps(num_inference_steps)"""
    if strength < 0 or strength > 1:
        raise ValueError(strength)
    scheduler.set_timesteps(num_inference_steps)
    offset = getattr(scheduler.config, "steps_offset", 0)
    init_timestep = int(num_inference_steps * strength) + offset
    init_timestep = min(init_timestep, num_inference_steps)
    t_noise = scheduler.timesteps[-init_timestep]
    t_start = max(num_inference_steps - init_timestep + offset, 0)
    return t_start, int(t_noise)


def denoise_loop(unet, scheduler, init_latents, noise, ctx2, num_inference_steps, strength, guidance_scale=7.5, eta=0.0,
                 generator=None, mask=None):
    """From the (already sampled, scaled and batch-repeated) init latents and the init noise: add_noise to t_noise, the CFG loop
    over timesteps[t_start:], and with a keep-mask the masking step after every scheduler step."""
    t_start, t_noise = img2img_start(scheduler, num_inference_steps, strength)
    B = init_latents.shape[0]
    latents = scheduler.add_noise(init_latents, noise, torch.tensor([t_noise] * B))
    params = inspect.signature(scheduler.step).parameters
    extra = {k: v for k, v in (("eta", eta), ("generator", generator)) if k in params}
    for t in scheduler.timesteps[t_start:]:
        x2 = torch.cat([latents] * 2)
        x2 = scheduler.scale_model_input(x2, t)
        eps = R.cfg_combine(unet(x2, t, ctx2).sample, guidance_scale)
        latents = scheduler.step(eps, t, latents, **extra).prev_sample
        if mask is not None:
            proper = scheduler.add_noise(init_latents, noise, torch.tensor([int(t)]))
            latents = proper * mask + latents * (1 - mask)
    return latents


def pipeline(unet, vae, scheduler, image, ctx2, num_inference_steps, strength, posterior_noise, init_noise, guidance_scale=7.5,
             eta=0.0, generator=None, mask=None):
    """image (1 or B, 3, H, W) in [-1, 1] -> (images (B, 3, H, W) in [0, 1], final latents); posterior_noise has the encoder's batch, init_noise
    and mask (1 = keep) the latents' batch B = ctx2.shape[0] // 2"""
    B = ctx2.shape[0] // 2
    init = 0.18215 * vae.encode(image).latent_dist.sample(noise=posterior_noise)
    if init.shape[0] == 1:
        init = torch.cat([init] * B)
    lat = denoise_loop(unet, scheduler, init, init_noise, ctx2, num_inference_steps, strength, guidance_scale, eta, generator,
                       mask)
    return (vae.decode(lat / 0.18215).sample / 2 + 0.5).clamp(0, 1), lat
