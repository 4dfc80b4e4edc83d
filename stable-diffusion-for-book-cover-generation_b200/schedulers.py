"""Scheduler facades with the diffusers 0.7.2 surface the reference touches (SURVEY.md 8b):

    DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                  clip_sample=False, set_alpha_to_one=False)                 inference.py:386-387
    PNDMScheduler(..., skip_prk_steps=True)                                   utils.py:222-224
    DDPMScheduler.from_config(path, subfolder="scheduler").add_noise(...)     finetune_sd.py:335-336, 473

Host side: timestep tables and per-step scalar coefficients (fp64 from the fp32 abar table).
Device side: ONE fused kernel per step through the C ABI (b200sd_cfg_ancestral_step for DDIM and DDPM /
b200sd_cfg_plms_step / b200sd_cfg_sigma_step for LMS, Euler and Euler-ancestral / b200sd_add_noise).  `step_cfg` additionally fuses the pipeline's
classifier-free-guidance combine into the same kernel.

Ancestral sampling (DDPMScheduler.step, DDIMScheduler.step with eta > 0) follows diffusers 0.7.2's formulas; its noise is
drawn by `step_noise` from the caller's generator.  Whether that noise stream is bit-equal to diffusers' own draws (which
device, whether the 0.7.2 pipeline hands `generator` to `step`) is not claimed.
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace
from typing import Callable, NamedTuple

import numpy as np
import torch

from . import ops


class SchedulerOutput(SimpleNamespace):
    pass


class CapturedStep(NamedTuple):
    """How sampler.CapturedSampler runs one scheduler (`captured_step`): the rows of its device coefficient table (one per
    executed step), the number of noise rows `draw_noise` fills, the slots of its history ring (0 or 4), whether the UNet input
    is the latents divided by the row's in_div (sampler_scale_input), and the ops.*_table call that closes the step.  `buffers`
    names the sampler's buffers ("noise", "ring", "saved": PNDM's saved sample) that `step` takes after the latents, in its
    argument order."""
    rows: list
    n_noise: int
    ring_slots: int
    scale_input: bool
    step: Callable
    buffers: tuple


def _betas(num_train_timesteps, beta_start, beta_end, beta_schedule):
    if beta_schedule == "scaled_linear":
        return torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
    if beta_schedule == "linear":
        return torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    raise NotImplementedError(f"{beta_schedule} is not implemented")


class _SchedulerBase:
    _defaults: dict = {}

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear", **kw):
        cfg = dict(self._defaults)
        cfg.update(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                   beta_schedule=beta_schedule)
        unknown = set(kw) - set(self._defaults)
        if unknown:
            raise TypeError(f"{type(self).__name__}: unexpected config keys {sorted(unknown)}")
        cfg.update(kw)
        self.config = SimpleNamespace(**cfg)
        self.num_train_timesteps = num_train_timesteps
        self.betas = _betas(num_train_timesteps, beta_start, beta_end, beta_schedule)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self._ac = self.alphas_cumprod.double().tolist()
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(0, num_train_timesteps)[::-1].copy())
        self._tables = {}

    # -- diffusers config plumbing ---------------------------------------------------------
    @classmethod
    def from_config(cls, path_or_dict, subfolder=None, **overrides):
        if isinstance(path_or_dict, dict):
            cfg = dict(path_or_dict)
        else:
            p = path_or_dict if subfolder is None else os.path.join(path_or_dict, subfolder)
            with open(os.path.join(p, "scheduler_config.json")) as f:
                cfg = json.load(f)
        cfg = {k: v for k, v in cfg.items() if not k.startswith("_")}
        allowed = {"num_train_timesteps", "beta_start", "beta_end", "beta_schedule", *cls._defaults}
        cfg = {k: v for k, v in cfg.items() if k in allowed}
        cfg.update(overrides)
        return cls(**cfg)

    from_pretrained = from_config

    def save_config(self, path):
        os.makedirs(path, exist_ok=True)
        d = dict(vars(self.config), _class_name=type(self).__name__)
        with open(os.path.join(path, "scheduler_config.json"), "w") as f:
            json.dump(d, f, indent=2)

    save_pretrained = save_config

    # -- shared behaviour ------------------------------------------------------------------
    def scale_model_input(self, sample, timestep=None):
        return sample

    def _noise_tables(self, device):
        key = str(device)
        if key not in self._tables:
            ac = self.alphas_cumprod.double()
            self._tables[key] = (ac.sqrt().float().to(device), (1 - ac).sqrt().float().to(device))
        return self._tables[key]

    def add_noise(self, original_samples, noise, timesteps):
        """sqrt(abar[t]) x0 + sqrt(1 - abar[t]) eps with a per-sample timestep (App. B.1)."""
        if original_samples.shape != noise.shape:
            raise ValueError("original_samples and noise must have the same shape")
        timesteps = timesteps.to(device=original_samples.device, dtype=torch.int64).reshape(-1)
        if timesteps.numel() == 1 and original_samples.shape[0] != 1:
            timesteps = timesteps.expand(original_samples.shape[0])
        if timesteps.numel() != original_samples.shape[0]:
            raise ValueError("timesteps must have one entry per sample")
        sa, sb = self._noise_tables(original_samples.device)
        return ops.add_noise(original_samples.contiguous(), noise.contiguous(), timesteps.contiguous(), sa, sb)

    def _alpha_prev(self, prev_t):
        return self._ac[prev_t] if prev_t >= 0 else self._final_alpha

    def _check_step_args(self, model_output, sample):
        if self.num_inference_steps is None:
            raise ValueError("Number of inference steps is 'None', you need to run 'set_timesteps' after creating "
                             "the scheduler")
        if model_output.numel() != sample.numel():
            raise ValueError("model_output and sample must have the same number of elements")

    def _ancestral_step(self, eps_u, eps_c, sample, guidance, coefs, generator, out=None):
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noisy, clip = coefs
        z = step_noise(sample, generator) if noisy else None
        return ops.cfg_ancestral_step(eps_u, eps_c, sample.contiguous(), z, guidance, sa_t, sb_t, c_x0, c_x, c_e, c_z, clip,
                                      out=out)

    def img2img_start(self, num_inference_steps, strength):
        """set_timesteps(n), then where diffusers 0.7.2's img2img / legacy inpainting pipelines enter the schedule for `strength`:
        (t_start, t_noise).  The loop runs over timesteps[t_start:] (possibly empty) and the init latents are noised to
        t_noise = timesteps[-init_timestep] -- timesteps[0] when init_timestep is 0, as in 0.7.2."""
        if not 0 <= strength <= 1:
            raise ValueError(f"The value of strength should in [0.0, 1.0] but is {strength}")
        self.set_timesteps(num_inference_steps)
        offset = getattr(self.config, "steps_offset", 0)
        init_timestep = min(int(num_inference_steps * strength) + offset, num_inference_steps)
        t_noise = int(self.timesteps[-init_timestep])
        return max(num_inference_steps - init_timestep + offset, 0), t_noise

    def ancestral_plan(self, eta=0.0, start=0):
        """One row per timestep of timesteps[start:] for b200sd_cfg_ancestral_step_table: sa_t sb_t c_x0 c_x c_e c_z noise_row
        clip, where noise_row counts the executed steps that add noise (the order step_noise draws them in) and is -1 on a step
        that adds none.  Returns (rows, number of noise rows)."""
        if self.num_inference_steps is None:
            raise ValueError("call set_timesteps first")
        rows, k = [], 0
        for t in self.timesteps.tolist()[start:]:
            sa_t, sb_t, c_x0, c_x, c_e, c_z, noisy, clip = self._ancestral_coefs(t, eta)
            rows.append([sa_t, sb_t, c_x0, c_x, c_e, c_z, float(k if noisy else -1), float(clip)])
            k += noisy
        return rows, k

    def captured_step(self, eta=0.0, start=0, inpaint=False):
        """CapturedSampler's step for DDIM (any eta) and DDPM over timesteps[start:]: ancestral_plan's rows, its noise table.
        Legacy inpainting (`inpaint`) adds a blend after the step and changes nothing here."""
        rows, n_noise = self.ancestral_plan(eta, start)
        return CapturedStep(rows, n_noise, 0, False, ops.cfg_ancestral_step_table, ("noise",))


def step_noise(sample, generator=None, out=None):
    """The noise of one stochastic step (DDPMScheduler.step, DDIMScheduler.step with eta > 0, and the captured sampler's
    noise table): torch.randn(sample.shape, float32) from `generator` on the generator's device (the sample's when generator is
    None), copied to the sample's device (or into `out`).  Steps draw in step order, and only steps that add noise draw."""
    dev = generator.device if generator is not None else sample.device
    z = torch.randn(tuple(sample.shape), generator=generator, dtype=torch.float32, device=dev)
    if out is None:
        if z.device == sample.device:
            return z
        out = torch.empty(z.shape, dtype=torch.float32, device=sample.device)
    return out.copy_(z)


class DDPMScheduler(_SchedulerBase):
    """The training-time surface the reference uses (add_noise / num_train_timesteps) and ancestral sampling, the scheduler
    finetune_sd.py:517-537 saves with its pipeline.  set_timesteps / step follow diffusers 0.7.2's formulas, including its
    previous-timestep rule abar[t - 1] at every step count.  Only `fixed_small` and `fixed_large` variances: the learned
    ones need an 8-channel UNet output that SD v1.x does not have."""
    _defaults = dict(trained_betas=None, variance_type="fixed_small", clip_sample=True)

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self._b = self.betas.double().tolist()
        self._a = self.alphas.double().tolist()

    def set_timesteps(self, num_inference_steps, device=None):
        if num_inference_steps < 1:
            raise ValueError("num_inference_steps out of range")
        if self.config.variance_type not in ("fixed_small", "fixed_large"):
            raise NotImplementedError(f"variance_type={self.config.variance_type!r} is not implemented")
        self.num_inference_steps = min(self.num_train_timesteps, num_inference_steps)
        ts = np.arange(0, self.num_train_timesteps, self.num_train_timesteps // self.num_inference_steps)[::-1]
        self.timesteps = torch.from_numpy(ts.copy().astype(np.int64))

    def _ancestral_coefs(self, timestep, eta=0.0):
        """(sa_t, sb_t, c_x0, c_x, c_e, c_z, adds_noise, clip) of one step, fp64 from the fp32 tables"""
        t = int(timestep)
        a_t = self._ac[t]
        a_p = self._ac[t - 1] if t > 0 else 1.0
        b_t, b_p = 1 - a_t, 1 - a_p
        c_x0 = a_p ** 0.5 * self._b[t] / b_t
        c_x = self._a[t] ** 0.5 * b_p / b_t
        c_z = 0.0
        if t > 0:
            if self.config.variance_type == "fixed_small":
                var = max(b_p / b_t * self._b[t], 1e-20)
            elif self.config.variance_type == "fixed_large":
                var = self._b[t]
            else:
                raise NotImplementedError(f"variance_type={self.config.variance_type!r} is not implemented")
            c_z = var ** 0.5
        return a_t ** 0.5, b_t ** 0.5, c_x0, c_x, 0.0, c_z, t > 0, bool(self.config.clip_sample)

    def step(self, model_output, timestep, sample, generator=None, return_dict: bool = True):
        self._check_step_args(model_output, sample)
        prev = self._ancestral_step(model_output.contiguous(), None, sample, 0.0, self._ancestral_coefs(timestep), generator)
        return SchedulerOutput(prev_sample=prev) if return_dict else (prev,)

    def step_cfg(self, model_output_2b, timestep, sample, guidance_scale, out=None, generator=None):
        """Fused `eps_u + s (eps_c - eps_u)` + DDPM update; model_output_2b is the (2B, ...) UNet output."""
        B = sample.shape[0]
        self._check_step_args(model_output_2b[:B], sample)
        prev = self._ancestral_step(model_output_2b[:B], model_output_2b[B:], sample, guidance_scale,
                                    self._ancestral_coefs(timestep), generator, out=out)
        return SchedulerOutput(prev_sample=prev)


class DDIMScheduler(_SchedulerBase):
    _defaults = dict(trained_betas=None, clip_sample=True, set_alpha_to_one=True, steps_offset=0)

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self._final_alpha = 1.0 if self.config.set_alpha_to_one else self._ac[0]
        self.final_alpha_cumprod = torch.tensor(self._final_alpha, dtype=torch.float32)
        if self.config.clip_sample:
            raise NotImplementedError("clip_sample=True is not on the reference path (inference.py:386-387)")

    def set_timesteps(self, num_inference_steps, device=None):
        if num_inference_steps > self.num_train_timesteps or num_inference_steps < 1:
            raise ValueError("num_inference_steps out of range")
        self.num_inference_steps = num_inference_steps
        ratio = self.num_train_timesteps // num_inference_steps
        ts = (np.arange(0, num_inference_steps) * ratio).round()[::-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(ts + self.config.steps_offset)

    def _ancestral_coefs(self, timestep, eta=0.0):
        """diffusers 0.7.2: sigma = eta sqrt((1 - a_p) / (1 - a_t) (1 - a_t / a_p)), x' = sqrt(a_p) x0 + sqrt(1 - a_p - sigma^2)
        eps + sigma z, with noise drawn on every step when eta > 0.  At eta = 0 this is the deterministic DDIM update
        sqrt(a_p) x0 + sqrt(1 - a_p) eps.  fp64 from the fp32 abar table."""
        if not 0.0 <= eta <= 1.0:
            raise ValueError(f"eta must be in [0, 1], got {eta}")
        t = int(timestep)
        prev_t = t - self.num_train_timesteps // self.num_inference_steps
        a_t, a_p = self._ac[t], self._alpha_prev(prev_t)
        var = (1 - a_p) / (1 - a_t) * (1 - a_t / a_p)
        sigma = eta * var ** 0.5
        return a_t ** 0.5, (1 - a_t) ** 0.5, a_p ** 0.5, 0.0, (1 - a_p - sigma ** 2) ** 0.5, sigma, eta > 0, False

    def step(self, model_output, timestep, sample, eta: float = 0.0, return_dict: bool = True, generator=None, **kw):
        self._check_step_args(model_output, sample)
        prev = self._ancestral_step(model_output.contiguous(), None, sample, 0.0, self._ancestral_coefs(timestep, eta), generator)
        return SchedulerOutput(prev_sample=prev) if return_dict else (prev,)

    def step_cfg(self, model_output_2b, timestep, sample, guidance_scale, out=None, eta: float = 0.0, generator=None):
        """Fused `eps_u + s (eps_c - eps_u)` + DDIM update; model_output_2b is the (2B, ...) UNet output."""
        B = sample.shape[0]
        self._check_step_args(model_output_2b[:B], sample)
        prev = self._ancestral_step(model_output_2b[:B], model_output_2b[B:], sample, guidance_scale,
                                    self._ancestral_coefs(timestep, eta), generator, out=out)
        return SchedulerOutput(prev_sample=prev)


class PNDMScheduler(_SchedulerBase):
    _defaults = dict(trained_betas=None, skip_prk_steps=False, set_alpha_to_one=False, steps_offset=0)

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        if not self.config.skip_prk_steps:
            raise NotImplementedError("only PLMS (skip_prk_steps=True) is on the reference path (utils.py:222-224)")
        self._final_alpha = 1.0 if self.config.set_alpha_to_one else self._ac[0]
        self.final_alpha_cumprod = torch.tensor(self._final_alpha, dtype=torch.float32)
        self.pndm_order = 4
        self.ets, self.counter, self.cur_sample = [], 0, None

    def set_timesteps(self, num_inference_steps, device=None):
        self.num_inference_steps = num_inference_steps
        ratio = self.num_train_timesteps // num_inference_steps
        _t = (np.arange(0, num_inference_steps) * ratio).round() + self.config.steps_offset
        plms = np.concatenate([_t[:-1], _t[-2:-1], _t[-1:]])[::-1].copy()
        self.timesteps = torch.from_numpy(plms.astype(np.int64))
        self.ets, self.counter, self.cur_sample = [], 0, None

    def _plms_call(self, counter, timestep, ets):
        """diffusers' step_plms (skip_prk_steps=True) for call number `counter` at `timestep`, given `ets`, the eps history
        kept so far (tensors for `_plms`, ring slots for `plms_plan`).  Returns (ets, keep_eps, w, hist, cx, ce, save_x,
        from_saved): ets trimmed to the entries later calls may read; whether this call's eps joins the history; the weights
        of this call's eps and of the history entries `hist` (newest first); cx, ce of _get_prev_sample; whether this call's
        sample is saved (the first call) or the saved sample is the one updated (the second call re-does the first timestep)."""
        t = int(timestep)
        ratio = self.num_train_timesteps // self.num_inference_steps
        prev_t = t - ratio
        keep_eps = counter != 1
        if keep_eps:
            ets = ets[-3:]
            n_after = len(ets) + 1
        else:
            prev_t, t = t, t + ratio
            n_after = len(ets)
        save_x = from_saved = False
        if n_after == 1 and counter == 0:
            w, hist, save_x = [1.0], [], True
        elif n_after == 1 and counter == 1:
            w, hist, from_saved = [0.5, 0.5], [ets[-1]], True
        elif n_after == 2:
            w, hist = [1.5, -0.5], [ets[-1]]
        elif n_after == 3:
            w, hist = [23 / 12, -16 / 12, 5 / 12], [ets[-1], ets[-2]]
        else:
            w, hist = [55 / 24, -59 / 24, 37 / 24, -9 / 24], [ets[-1], ets[-2], ets[-3]]
        a_t, a_p = self._ac[t], self._alpha_prev(prev_t)
        b_t, b_p = 1 - a_t, 1 - a_p
        cx = (a_p / a_t) ** 0.5
        ce = (a_p - a_t) / (a_t * b_p ** 0.5 + (a_t * b_t * a_p) ** 0.5)
        return ets, keep_eps, w, hist, cx, ce, save_x, from_saved

    def _plms(self, eps_u, eps_c, timestep, sample, guidance, out=None):
        self._check_step_args(eps_u, sample)
        self.ets, keep_eps, w, hist, cx, ce, save_x, from_saved = self._plms_call(self.counter, timestep, self.ets)
        x = sample
        if save_x:
            self.cur_sample = sample.clone()    # the caller may recycle its latent buffers (step_cfg(out=...))
        elif from_saved:
            x, self.cur_sample = self.cur_sample, None
        eps_out = torch.empty_like(eps_u) if keep_eps else None
        if eps_u.dtype == torch.float16:      # fp16 pipelines: the eps history is kept in fp32
            eps_u, eps_c = eps_u.float(), (None if eps_c is None else eps_c.float())
            eps_out = torch.empty_like(eps_u) if keep_eps else None
            prev = ops.cfg_plms_step(eps_u, eps_c, x.float().contiguous(), hist, w, guidance, cx, ce, eps_out=eps_out).to(x.dtype)
            if out is not None:
                prev = out.copy_(prev)
        else:
            prev = ops.cfg_plms_step(eps_u, eps_c, x.contiguous(), hist, w, guidance, cx, ce, out=out, eps_out=eps_out)
        if keep_eps:
            self.ets.append(eps_out)
        self.counter += 1
        return SchedulerOutput(prev_sample=prev)

    def plms_plan(self, start=0):
        """The whole call sequence of one sampling run over timesteps[start:] as data: one row per UNet call for
        b200sd_cfg_plms_step_table (w0 w1 w2 w3 | cx ce | ring slots of ets[-1], ets[-2], ets[-3] | slot this call's eps goes to |
        x_from_saved | save_x).  It is `_plms_call` run once on the host with a 4-slot eps ring instead of tensors, so that
        sampler.CapturedSampler can replay every call as the same CUDA graph (the step index lives on the device).  The call
        counter starts at 0 on timesteps[start], as the per-call loop's does after set_timesteps."""
        if self.num_inference_steps is None:
            raise ValueError("call set_timesteps first")
        rows, ets = [], []
        for counter, timestep in enumerate(self.timesteps.tolist()[start:]):
            ets, keep_eps, w, hist, cx, ce, save_x, from_saved = self._plms_call(counter, timestep, ets)
            slot = -1
            if keep_eps:
                slot = next(k for k in range(4) if k not in ets)       # ets holds <= 3 live slots here
                ets.append(slot)
            rows.append(w + [0.0] * (4 - len(w)) + [cx, ce] + [float(h) for h in hist] + [-1.0] * (3 - len(hist))
                        + [float(slot), float(from_saved), float(save_x)])
        return rows

    def captured_step(self, eta=0.0, start=0, inpaint=False):
        """PLMS over timesteps[start:]: plms_plan's rows, the 4-slot eps ring and the sample saved by the first call"""
        return CapturedStep(self.plms_plan(start), 0, 4, False, ops.cfg_plms_step_table, ("saved", "ring"))

    def step(self, model_output, timestep, sample, return_dict: bool = True, **kw):
        out = self._plms(model_output.contiguous(), None, timestep, sample, 0.0)
        return out if return_dict else (out.prev_sample,)

    def step_cfg(self, model_output_2b, timestep, sample, guidance_scale, out=None):
        B = sample.shape[0]
        return self._plms(model_output_2b[:B], model_output_2b[B:], timestep, sample, guidance_scale, out=out)


# ---------------------------------------------------------------------------------------------------
# The sigma-space family of diffusers 0.7.2 (scheduling_lms_discrete.py, scheduling_euler_discrete.py,
# scheduling_euler_ancestral_discrete.py).  They sample the variance-exploding ODE x_VE = x_VP / sqrt(abar): the UNet input is
# scaled by 1 / sqrt(sigma^2 + 1) and the timesteps are fractional.  One step rule (`_sigma_call`) serves the per-call step and
# the captured sampler's table (`sigma_plan`); the device work is one fused kernel, b200sd_cfg_sigma_step.
# ---------------------------------------------------------------------------------------------------
class _SigmaSchedulerBase(_SchedulerBase):
    """sigmas = ((1 - abar) / abar) ** 0.5 in fp32; set_timesteps(n): timesteps = linspace(0, T - 1, n)[::-1] (float64), sigmas
    interpolated at them plus a final 0, fp32.  A timestep is looked up by exact match in `timesteps`."""
    _defaults = dict(trained_betas=None)
    _keeps_history = False

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        T = self.num_train_timesteps
        self._train_sigmas = (((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5).numpy()
        self.sigmas = torch.from_numpy(np.concatenate([self._train_sigmas[::-1], [0.0]]).astype(np.float32))
        self.init_noise_sigma = float(self.sigmas.max())
        self._set_schedule(np.linspace(0, T - 1, T, dtype=float)[::-1].copy(), self.sigmas)
        self.num_inference_steps = None

    def _set_schedule(self, timesteps, sigmas):
        self.timesteps = torch.from_numpy(timesteps)
        self.sigmas = sigmas
        self._sig = sigmas.numpy()
        self._step_index = {t: i for i, t in enumerate(timesteps.tolist())}
        self._in_div = (sigmas ** 2 + 1) ** 0.5           # fp32, as scale_model_input computes it
        self._in_div_dev = {}
        self._lms_cache = {}
        self._derivs = []

    def set_timesteps(self, num_inference_steps, device=None):
        if num_inference_steps < 1:
            raise ValueError("num_inference_steps out of range")
        self.num_inference_steps = num_inference_steps
        T = self.num_train_timesteps
        ts = np.linspace(0, T - 1, num_inference_steps, dtype=float)[::-1].copy()
        sig = np.interp(ts, np.arange(0, len(self._train_sigmas)), self._train_sigmas)
        self._set_schedule(ts, torch.from_numpy(np.concatenate([sig, [0.0]]).astype(np.float32)))

    def _index(self, timestep):
        i = self._step_index.get(float(timestep))
        if i is None:
            raise ValueError(f"timestep {float(timestep)!r} is not in this scheduler's timesteps")
        return i

    def scale_model_input(self, sample, timestep):
        """sample / ((sigma ** 2 + 1) ** 0.5): a true division by a tensor on the sample's device"""
        i = self._index(timestep)
        key = str(sample.device)
        if key not in self._in_div_dev:
            self._in_div_dev[key] = self._in_div.to(sample.device)
        return sample / self._in_div_dev[key][i]

    def add_noise(self, original_samples, noise, timesteps):
        raise NotImplementedError(f"{type(self).__name__}.add_noise (sigma-space noising) is not implemented")

    def img2img_start(self, num_inference_steps, strength):
        # 0.7.2 noises the init latents in sigma space here; add_noise and the inpainting blend index integer timesteps
        raise NotImplementedError(f"image-to-image and inpainting with {type(self).__name__} are not implemented")

    # -- the step rule ----------------------------------------------------------------------------
    def _coefs(self, i, order, sig):
        """(weights of [d, d[-1], ...], adds noise, sigma_up) of step i"""
        raise NotImplementedError

    def _sigma_call(self, i, hist, order=4, sig=None):
        """The decisions of step index i given `hist`, the derivatives kept by earlier steps (tensors for the per-call step, ring
        slots for `sigma_plan`), oldest first.  Returns (hist, sigma, coefs, used, keep_d, noisy, sigma_up): hist trimmed to the
        entries this and later steps may read; the weights `coefs` of this step's derivative and of the history entries `used`
        (newest first); whether this step's derivative joins the history; whether it adds sigma_up * z.  `sig` (default: this
        schedule's fp32 sigmas) may be another sigma sequence, e.g. in float64."""
        if not 1 <= order <= 4:
            raise ValueError(f"order must be in 1..4, got {order}")
        sig = self._sig if sig is None else sig
        coefs, noisy, sigma_up = self._coefs(i, order, sig)
        keep = self._keeps_history and order > 1
        hist = list(hist)[max(0, len(hist) - (order - 1)):] if keep else []
        used = hist[::-1][:len(coefs) - 1]
        return hist, sig[i], coefs[:len(used) + 1], used, keep, noisy, sigma_up

    def sigma_plan(self, order=4):
        """The whole run as rows for b200sd_cfg_sigma_step_table: sigma | c0 c1 c2 c3 | h1 h2 h3 (ring slots, -1 unused) |
        out_slot | noise_row (-1 none) | sigma_up | in_div.  `_sigma_call` run once on the host with a 4-slot ring instead of
        tensors; noise rows are numbered in step order, as the per-call step draws.  Returns (rows, number of noise rows)."""
        if self.num_inference_steps is None:
            raise ValueError("call set_timesteps first")
        rows, hist, k = [], [], 0
        for i in range(len(self.timesteps)):
            hist, sigma, coefs, used, keep, noisy, sigma_up = self._sigma_call(i, hist, order)
            slot = next(s for s in range(4) if s not in hist) if keep else -1
            rows.append([float(sigma)] + [float(c) for c in coefs] + [0.0] * (4 - len(coefs))
                        + [float(h) for h in used] + [-1.0] * (3 - len(used))
                        + [float(slot), float(k if noisy else -1), float(sigma_up), float(self._in_div[i])])
            if keep:
                hist.append(slot)
            k += noisy
        return rows, k

    def captured_step(self, eta=0.0, start=0, inpaint=False):
        """The full schedule only: sigma_plan's rows, the derivative ring of LMS, the noise table of Euler-ancestral, and the
        UNet input divided by in_div"""
        if start != 0 or inpaint:
            raise ValueError(f"{type(self).__name__}: image-to-image and inpainting (start != 0, inpaint=True) are not "
                             "implemented for the sigma-space schedulers")
        rows, n_noise = self.sigma_plan()
        return CapturedStep(rows, n_noise, 4 if self._keeps_history else 0, True, ops.cfg_sigma_step_table, ("ring", "noise"))

    def _sigma_step(self, eps_u, eps_c, timestep, sample, guidance, generator=None, out=None, order=4):
        self._check_step_args(eps_u, sample)
        i = self._index(timestep)
        self._derivs, sigma, coefs, used, keep, noisy, sigma_up = self._sigma_call(i, self._derivs, order)
        if eps_u.dtype == torch.float16:      # fp16 pipelines: computed in fp32, the result cast back
            eps_u, eps_c = eps_u.float(), (None if eps_c is None else eps_c.float())
        x = sample.float().contiguous()
        z = step_noise(x, generator) if noisy else None
        d = torch.empty_like(x) if keep else None
        fits = out is not None and out.dtype == torch.float32 and out.is_contiguous()
        prev = ops.cfg_sigma_step(eps_u.contiguous(), None if eps_c is None else eps_c.contiguous(), x, guidance, sigma, coefs,
                                  used, z, sigma_up, out=out if fits else None, d_out=d)
        if keep:
            self._derivs.append(d)
        if out is not None and not fits:
            prev = out.copy_(prev)
        elif prev.dtype != sample.dtype:
            prev = prev.to(sample.dtype)
        return SchedulerOutput(prev_sample=prev)


def _lms_coefficient(sig, order, t, current_order):
    """0.7.2's get_lms_coefficient: the integral of the Lagrange basis polynomial over [sigma[t], sigma[t + 1]], with the
    integrand evaluated in sig's precision (fp32 there: the sigmas are fp32 tensors)"""
    from scipy import integrate

    def lms_derivative(tau):
        prod = 1.0
        for k in range(order):
            if current_order == k:
                continue
            prod *= (tau - sig[t - k]) / (sig[t - current_order] - sig[t - k])
        return prod

    return integrate.quad(lms_derivative, float(sig[t]), float(sig[t + 1]), epsrel=1e-4)[0]


class LMSDiscreteScheduler(_SigmaSchedulerBase):
    """diffusers 0.7.2 LMSDiscreteScheduler: linear multistep of order min(step index + 1, order) over the ODE derivatives."""
    _keeps_history = True

    def _coefs(self, i, order, sig):
        o = min(i + 1, order)
        if sig is not self._sig:
            return [_lms_coefficient(sig, o, i, k) for k in range(o)], False, 0.0
        key = (o, i)
        if key not in self._lms_cache:
            self._lms_cache[key] = [_lms_coefficient(sig, o, i, k) for k in range(o)]
        return self._lms_cache[key], False, 0.0

    def step(self, model_output, timestep, sample, order: int = 4, return_dict: bool = True):
        out = self._sigma_step(model_output, None, timestep, sample, 0.0, order=order)
        return out if return_dict else (out.prev_sample,)

    def step_cfg(self, model_output_2b, timestep, sample, guidance_scale, out=None, order: int = 4):
        """Fused `eps_u + s (eps_c - eps_u)` + LMS update; model_output_2b is the (2B, ...) UNet output."""
        B = sample.shape[0]
        return self._sigma_step(model_output_2b[:B], model_output_2b[B:], timestep, sample, guidance_scale, out=out, order=order)


class EulerDiscreteScheduler(_SigmaSchedulerBase):
    """diffusers 0.7.2 EulerDiscreteScheduler with s_churn = 0 (x' = x + (sigma_next - sigma) d).  It draws no noise; 0.7.2
    draws a tensor it does not use on every step, so the generator's state afterwards differs from diffusers'."""

    def _coefs(self, i, order, sig):
        return [sig[i + 1] - sig[i]], False, 0.0

    def _check_churn(self, timestep, s_churn, s_tmin, s_tmax):
        sigma = float(self._sig[self._index(timestep)])
        gamma = min(s_churn / (len(self._sig) - 1), 2 ** 0.5 - 1) if s_tmin <= sigma <= s_tmax else 0.0
        if gamma > 0:
            raise NotImplementedError("EulerDiscreteScheduler with s_churn > 0 is not implemented")

    def step(self, model_output, timestep, sample, s_churn: float = 0.0, s_tmin: float = 0.0, s_tmax: float = float("inf"),
             s_noise: float = 1.0, generator=None, return_dict: bool = True):
        self._check_churn(timestep, s_churn, s_tmin, s_tmax)
        out = self._sigma_step(model_output, None, timestep, sample, 0.0)
        return out if return_dict else (out.prev_sample,)

    def step_cfg(self, model_output_2b, timestep, sample, guidance_scale, out=None, s_churn: float = 0.0, s_tmin: float = 0.0,
                 s_tmax: float = float("inf"), s_noise: float = 1.0, generator=None):
        """Fused `eps_u + s (eps_c - eps_u)` + Euler update; model_output_2b is the (2B, ...) UNet output."""
        self._check_churn(timestep, s_churn, s_tmin, s_tmax)
        B = sample.shape[0]
        return self._sigma_step(model_output_2b[:B], model_output_2b[B:], timestep, sample, guidance_scale, out=out)


class EulerAncestralDiscreteScheduler(_SigmaSchedulerBase):
    """diffusers 0.7.2 EulerAncestralDiscreteScheduler: x' = x + (sigma_down - sigma) d + sigma_up z with
    sigma_up = (sigma_to^2 (sigma_from^2 - sigma_to^2) / sigma_from^2) ** 0.5, sigma_down = (sigma_to^2 - sigma_up^2) ** 0.5.
    Every step, the last one included (sigma_up = 0 there), draws one `step_noise` from the caller's generator."""

    def _coefs(self, i, order, sig):
        sf, st = sig[i], sig[i + 1]
        sigma_up = np.sqrt(st * st * (sf * sf - st * st) / (sf * sf))
        sigma_down = np.sqrt(st * st - sigma_up * sigma_up)
        return [sigma_down - sf], True, sigma_up

    def step(self, model_output, timestep, sample, generator=None, return_dict: bool = True):
        out = self._sigma_step(model_output, None, timestep, sample, 0.0, generator=generator)
        return out if return_dict else (out.prev_sample,)

    def step_cfg(self, model_output_2b, timestep, sample, guidance_scale, out=None, generator=None):
        """Fused `eps_u + s (eps_c - eps_u)` + Euler-ancestral update; model_output_2b is the (2B, ...) UNet output."""
        B = sample.shape[0]
        return self._sigma_step(model_output_2b[:B], model_output_2b[B:], timestep, sample, guidance_scale, generator=generator,
                                out=out)


SCHEDULERS = (DDIMScheduler, PNDMScheduler, DDPMScheduler, LMSDiscreteScheduler, EulerDiscreteScheduler,
              EulerAncestralDiscreteScheduler)
