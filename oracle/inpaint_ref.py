"""ORACLE (test infrastructure, not product code) -- diffusers 0.7.2's StableDiffusionInpaintPipeline (the 9-channel inpainting
UNet) restated in plain fp32 PyTorch + numpy, on the oracle UNet (`make_oracle_unet(in_channels=9)`), VAE and schedulers
(oracle.unet_ref, oracle.vae_ref, oracle.schedulers_ref, oracle.ancestral_ref, oracle.sigma_ref).

diffusers is not installed here and its source is not in the tree: the 0.7.2 behaviour below is written from the release's
pipeline_stable_diffusion_inpaint.py as the maintainer remembers it.  The quirks kept:
  * prepare_mask_and_masked_image: the image is not resized ("RGB" -> NCHW -> / 127.5 - 1); the mask ("L" -> / 255) is
    binarised at 0.5 and NOT inverted (1 = repaint); masked_image = image * (mask < 0.5).
  * the mask goes to latent size with F.interpolate's default mode (nearest), not PIL's resampling.
  * every step concatenates [latents | mask | masked-image latents] BEFORE scale_model_input, so the sigma-space schedulers
    divide the mask and the masked latents by (sigma^2 + 1)^0.5 too (later diffusers releases scale first).
  * there is no `strength`: the run starts from pure noise over the full schedule.

Every random draw is an explicit argument (the initial latents, the posterior noise of the masked image; the step noise comes
from `generator` as in ancestral_ref / sigma_ref), so tests can feed the product and the oracle identical draws.  No published
known answer of this pipeline exists, so none is claimed.
"""
from __future__ import annotations

import inspect

import numpy as np
import torch
import torch.nn.functional as F

from . import schedulers_ref as R


def prepare_mask_and_masked_image(image, mask):
    """PIL image and mask -> (mask (1, 1, H, W) in {0, 1}, masked_image (1, 3, H, W))"""
    image = np.array(image.convert("RGB"))
    image = image[None].transpose(0, 3, 1, 2)
    image = torch.from_numpy(image).to(dtype=torch.float32) / 127.5 - 1.0

    mask = np.array(mask.convert("L"))
    mask = mask.astype(np.float32) / 255.0
    mask = mask[None, None]
    mask[mask < 0.5] = 0
    mask[mask >= 0.5] = 1
    mask = torch.from_numpy(mask)

    masked_image = image * (mask < 0.5)
    return mask, masked_image


def latent_mask(mask, h, w):
    """the pipeline's mask at latent size: F.interpolate(mask, size=(h, w)), torch's default mode"""
    return F.interpolate(mask, size=(h, w))


def denoise_loop(unet, scheduler, latents, mask, masked_image_latents, ctx2, num_inference_steps=50, guidance_scale=7.5, eta=0.0,
                 generator=None):
    """The 0.7.2 loop: latents * init_noise_sigma; per step cat([latents] * 2), cat with cat([mask] * 2) and
    cat([masked_image_latents] * 2) along the channels, then scale_model_input; `eta` / `generator` only to a step that takes
    them.  mask (B, 1, h, w) and masked_image_latents (B, 4, h, w) already have the latents' batch."""
    params = inspect.signature(scheduler.step).parameters
    extra = {k: v for k, v in (("eta", eta), ("generator", generator)) if k in params}
    if 4 + mask.shape[1] + masked_image_latents.shape[1] != unet.in_channels:
        raise ValueError("the UNet does not take latents | mask | masked-image latents")
    scheduler.set_timesteps(num_inference_steps)
    mask2 = torch.cat([mask] * 2)
    masked2 = torch.cat([masked_image_latents] * 2)
    latents = latents * scheduler.init_noise_sigma
    for t in scheduler.timesteps:
        x = torch.cat([latents] * 2)
        x = torch.cat([x, mask2, masked2], dim=1)
        x = scheduler.scale_model_input(x, t)
        eps = R.cfg_combine(unet(x, t, ctx2).sample, guidance_scale)
        latents = scheduler.step(eps, t, latents, **extra).prev_sample
    return latents


def pipeline(unet, vae, scheduler, mask, masked_image, ctx2, num_inference_steps, init_latents, posterior_noise,
             guidance_scale=7.5, eta=0.0, generator=None):
    """mask (1|B, 1, H, W) and masked_image (1|B, 3, H, W) as prepare_mask_and_masked_image returns them -> (images (B, 3, H, W)
    in [0, 1], final latents).  init_latents (B, 4, H/8, W/8) is the pipeline's first draw, posterior_noise (the masked image's
    batch) its second."""
    B = ctx2.shape[0] // 2
    h, w = init_latents.shape[2:]
    m = latent_mask(mask, h, w)
    masked_latents = 0.18215 * vae.encode(masked_image).latent_dist.sample(noise=posterior_noise)
    m = m.expand(B, -1, -1, -1) if m.shape[0] == 1 else m
    masked_latents = masked_latents.expand(B, -1, -1, -1) if masked_latents.shape[0] == 1 else masked_latents
    lat = denoise_loop(unet, scheduler, init_latents, m, masked_latents, ctx2, num_inference_steps, guidance_scale, eta, generator)
    return (vae.decode(lat / 0.18215).sample / 2 + 0.5).clamp(0, 1), lat
