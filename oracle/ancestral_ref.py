"""ORACLE (test infrastructure, not product code) -- diffusers 0.7.2's ancestral samplers restated in plain fp32 PyTorch:
DDPMScheduler.set_timesteps / step (scheduling_ddpm.py) and the eta > 0 branch of DDIMScheduler.step (scheduling_ddim.py),
with the same `alphas_cumprod` tensors, `** 0.5` and order of operations.  Built on top of oracle.schedulers_ref; its
eta = 0 paths are called unchanged.

Reference call sites: the pipeline `finetune_sd.py:517-537` saves with `scheduler=noise_scheduler` (a DDPMScheduler) and
`load_model` (`utils.py:187-191`) samples with after training.  No published known answer of diffusers is transcribed for
these: the DDPM == DDIM(eta = 1) equivalence at 1000 steps ties the two restatements together (tests/test_ancestral_host.py).
"""
from __future__ import annotations

import inspect
from types import SimpleNamespace

import numpy as np
import torch

from . import schedulers_ref as R


def step_noise(model_output, generator=None):
    """The noise of one stochastic step: torch.randn(shape, float32) from `generator` on the generator's device (the
    model output's when generator is None), moved to the model output's device."""
    dev = generator.device if generator is not None else model_output.device
    return torch.randn(tuple(model_output.shape), generator=generator, dtype=torch.float32, device=dev).to(model_output.device)


class DDPMSchedulerRef(R.DDPMSchedulerRef):
    """scheduling_ddpm.py: set_timesteps / step / _get_variance (fixed_small, fixed_large)."""

    def __init__(self, variance_type="fixed_small", clip_sample=True, **kw):
        super().__init__(variance_type=variance_type, clip_sample=clip_sample, **kw)
        self.one = torch.tensor(1.0)
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(0, self.num_train_timesteps)[::-1].copy())

    def set_timesteps(self, num_inference_steps, device=None):
        num_inference_steps = min(self.config.num_train_timesteps, num_inference_steps)
        self.num_inference_steps = num_inference_steps
        timesteps = np.arange(0, self.config.num_train_timesteps,
                              self.config.num_train_timesteps // self.num_inference_steps)[::-1].copy()
        self.timesteps = torch.from_numpy(timesteps)

    def _get_variance(self, t):
        alpha_prod_t = self.alphas_cumprod[t]
        alpha_prod_t_prev = self.alphas_cumprod[t - 1] if t > 0 else self.one
        variance = (1 - alpha_prod_t_prev) / (1 - alpha_prod_t) * self.betas[t]
        if self.config.variance_type == "fixed_small":
            variance = torch.clamp(variance, min=1e-20)
        elif self.config.variance_type == "fixed_large":
            variance = self.betas[t]
        else:
            raise NotImplementedError(self.config.variance_type)
        return variance

    def coefficients(self, t):
        """(pred_original_sample_coeff, current_sample_coeff) of step 4 of 0.7.2's `step`"""
        alpha_prod_t = self.alphas_cumprod[t]
        alpha_prod_t_prev = self.alphas_cumprod[t - 1] if t > 0 else self.one
        beta_prod_t = 1 - alpha_prod_t
        beta_prod_t_prev = 1 - alpha_prod_t_prev
        pred_original_sample_coeff = (alpha_prod_t_prev ** (0.5) * self.betas[t]) / beta_prod_t
        current_sample_coeff = self.alphas[t] ** (0.5) * beta_prod_t_prev / beta_prod_t
        return pred_original_sample_coeff, current_sample_coeff

    def step(self, model_output, timestep, sample, generator=None):
        t = int(timestep)
        alpha_prod_t = self.alphas_cumprod[t]
        beta_prod_t = 1 - alpha_prod_t
        pred_original_sample = (sample - beta_prod_t ** (0.5) * model_output) / alpha_prod_t ** (0.5)
        if self.config.clip_sample:
            pred_original_sample = torch.clamp(pred_original_sample, -1, 1)
        pred_original_sample_coeff, current_sample_coeff = self.coefficients(t)
        pred_prev_sample = pred_original_sample_coeff * pred_original_sample + current_sample_coeff * sample
        variance = 0
        if t > 0:
            noise = step_noise(model_output, generator)
            variance = (self._get_variance(t) ** 0.5) * noise
        pred_prev_sample = pred_prev_sample + variance
        return SimpleNamespace(prev_sample=pred_prev_sample, pred_original_sample=pred_original_sample)


class DDIMSchedulerRef(R.DDIMSchedulerRef):
    """scheduling_ddim.py `step` with eta > 0 (use_clipped_model_output=False); eta = 0 is schedulers_ref's step as it is."""

    def _get_variance(self, timestep, prev_timestep):
        alpha_prod_t = self.alphas_cumprod[timestep]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        beta_prod_t = 1 - alpha_prod_t
        beta_prod_t_prev = 1 - alpha_prod_t_prev
        return (beta_prod_t_prev / beta_prod_t) * (1 - alpha_prod_t / alpha_prod_t_prev)

    def step(self, model_output, timestep, sample, eta: float = 0.0, generator=None):
        if eta == 0.0:
            return super().step(model_output, timestep, sample)
        t = int(timestep)
        prev_t = t - self.num_train_timesteps // self.num_inference_steps
        a_t = self.alphas_cumprod[t]
        a_p = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.final_alpha_cumprod
        b_t = 1 - a_t
        x0 = (sample - b_t ** 0.5 * model_output) / a_t ** 0.5
        if self.config.clip_sample:
            x0 = torch.clamp(x0, -1, 1)
        variance = self._get_variance(t, prev_t)
        std_dev_t = eta * variance ** (0.5)
        direction = (1 - a_p - std_dev_t ** 2) ** (0.5) * model_output
        prev = a_p ** (0.5) * x0 + direction
        noise = step_noise(model_output, generator)
        prev = prev + self._get_variance(t, prev_t) ** (0.5) * eta * noise
        return SimpleNamespace(prev_sample=prev, pred_original_sample=x0)


def denoise_loop(unet, scheduler, latents, ctx2, num_inference_steps=50, guidance_scale=7.5, eta=0.0, generator=None):
    """schedulers_ref.denoise_loop with `eta` and `generator`: as in diffusers, each goes only to a step that takes it."""
    params = inspect.signature(scheduler.step).parameters
    extra = {k: v for k, v in (("eta", eta), ("generator", generator)) if k in params}
    scheduler.set_timesteps(num_inference_steps)
    latents = latents * scheduler.init_noise_sigma
    for t in scheduler.timesteps:
        x2 = torch.cat([latents] * 2)
        x2 = scheduler.scale_model_input(x2, t)
        eps = unet(x2, t, ctx2).sample
        eps = R.cfg_combine(eps, guidance_scale)
        latents = scheduler.step(eps, t, latents, **extra).prev_sample
    return latents
