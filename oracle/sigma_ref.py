"""ORACLE (test infrastructure, not product code) -- diffusers 0.7.2's sigma-space schedulers restated in plain fp32 PyTorch:
LMSDiscreteScheduler (scheduling_lms_discrete.py), EulerDiscreteScheduler (scheduling_euler_discrete.py, s_churn = 0) and
EulerAncestralDiscreteScheduler (scheduling_euler_ancestral_discrete.py), with the same fp32 `sigmas` tensors -- inside the LMS
integrand too --, `** 0.5`, float64 timesteps and order of operations.  Built on oracle.schedulers_ref's base (betas and
alphas_cumprod), which is unchanged.

The noise of an Euler-ancestral step is passed through `generator` and drawn by oracle.ancestral_ref.step_noise, one draw per
step, the last one included.  Euler's unused per-step draw of 0.7.x is not restated (it does not change the result).
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import torch
from scipy import integrate

from . import schedulers_ref as R
from .ancestral_ref import step_noise


class _SigmaRef(R._Base):
    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear", **kw):
        super().__init__(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                         beta_schedule=beta_schedule, **kw)
        sigmas = np.array(((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5)
        sigmas = np.concatenate([sigmas[::-1], [0.0]]).astype(np.float32)
        self.sigmas = torch.from_numpy(sigmas)
        self.init_noise_sigma = self.sigmas.max()
        self.num_inference_steps = None
        timesteps = np.linspace(0, num_train_timesteps - 1, num_train_timesteps, dtype=float)[::-1].copy()
        self.timesteps = torch.from_numpy(timesteps)
        self.derivatives = []

    def set_timesteps(self, num_inference_steps, device=None):
        self.num_inference_steps = num_inference_steps
        timesteps = np.linspace(0, self.config.num_train_timesteps - 1, num_inference_steps, dtype=float)[::-1].copy()
        sigmas = np.array(((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5)
        sigmas = np.interp(timesteps, np.arange(0, len(sigmas)), sigmas)
        sigmas = np.concatenate([sigmas, [0.0]]).astype(np.float32)
        self.sigmas = torch.from_numpy(sigmas)
        self.timesteps = torch.from_numpy(timesteps)
        self.derivatives = []

    def _step_index(self, timestep):
        if isinstance(timestep, torch.Tensor):
            timestep = timestep.to(self.timesteps.device)
        return (self.timesteps == timestep).nonzero().item()

    def scale_model_input(self, sample, timestep):
        sigma = self.sigmas[self._step_index(timestep)]
        return sample / ((sigma ** 2 + 1) ** 0.5)


class LMSDiscreteSchedulerRef(_SigmaRef):
    def get_lms_coefficient(self, order, t, current_order):
        def lms_derivative(tau):
            prod = 1.0
            for k in range(order):
                if current_order == k:
                    continue
                prod *= (tau - self.sigmas[t - k]) / (self.sigmas[t - current_order] - self.sigmas[t - k])
            return float(prod)

        return integrate.quad(lms_derivative, float(self.sigmas[t]), float(self.sigmas[t + 1]), epsrel=1e-4)[0]

    def step(self, model_output, timestep, sample, order=4):
        step_index = self._step_index(timestep)
        sigma = self.sigmas[step_index]
        pred_original_sample = sample - sigma * model_output
        derivative = (sample - pred_original_sample) / sigma
        self.derivatives.append(derivative)
        if len(self.derivatives) > order:
            self.derivatives.pop(0)
        order = min(step_index + 1, order)
        lms_coeffs = [self.get_lms_coefficient(order, step_index, curr_order) for curr_order in range(order)]
        prev_sample = sample + sum(coeff * derivative for coeff, derivative in zip(lms_coeffs, reversed(self.derivatives)))
        return SimpleNamespace(prev_sample=prev_sample, pred_original_sample=pred_original_sample)


class EulerDiscreteSchedulerRef(_SigmaRef):
    def step(self, model_output, timestep, sample, s_churn=0.0, s_tmin=0.0, s_tmax=float("inf"), s_noise=1.0, generator=None):
        step_index = self._step_index(timestep)
        sigma = self.sigmas[step_index]
        gamma = min(s_churn / (len(self.sigmas) - 1), 2 ** 0.5 - 1) if s_tmin <= sigma <= s_tmax else 0.0
        assert gamma == 0.0, "oracle restates s_churn = 0 only"
        sigma_hat = sigma * (gamma + 1)
        pred_original_sample = sample - sigma_hat * model_output
        derivative = (sample - pred_original_sample) / sigma_hat
        dt = self.sigmas[step_index + 1] - sigma_hat
        prev_sample = sample + derivative * dt
        return SimpleNamespace(prev_sample=prev_sample, pred_original_sample=pred_original_sample)


class EulerAncestralDiscreteSchedulerRef(_SigmaRef):
    def step(self, model_output, timestep, sample, generator=None):
        step_index = self._step_index(timestep)
        sigma = self.sigmas[step_index]
        pred_original_sample = sample - sigma * model_output
        sigma_from = self.sigmas[step_index]
        sigma_to = self.sigmas[step_index + 1]
        sigma_up = (sigma_to ** 2 * (sigma_from ** 2 - sigma_to ** 2) / sigma_from ** 2) ** 0.5
        sigma_down = (sigma_to ** 2 - sigma_up ** 2) ** 0.5
        derivative = (sample - pred_original_sample) / sigma
        dt = sigma_down - sigma
        prev_sample = sample + derivative * dt
        noise = step_noise(model_output, generator)
        prev_sample = prev_sample + noise * sigma_up
        return SimpleNamespace(prev_sample=prev_sample, pred_original_sample=pred_original_sample)


def denoise_loop(unet, scheduler, latents, ctx2, num_inference_steps=50, guidance_scale=7.5, generator=None):
    """The 0.7.2 pipeline loop for these schedulers: latents * init_noise_sigma, scale_model_input before every UNet call (the
    UNet receives the float64 timestep tensor), `generator` only to a step that takes it (Euler-ancestral)."""
    import inspect
    extra = {"generator": generator} if "generator" in inspect.signature(scheduler.step).parameters else {}
    scheduler.set_timesteps(num_inference_steps)
    latents = latents * scheduler.init_noise_sigma
    for t in scheduler.timesteps:
        x2 = torch.cat([latents] * 2)
        x2 = scheduler.scale_model_input(x2, t)
        eps = unet(x2, t, ctx2).sample
        eps = R.cfg_combine(eps, guidance_scale)
        latents = scheduler.step(eps, t, latents, **extra).prev_sample
    return latents
