"""The whole denoising step of StableDiffusionPipeline.__call__ as ONE CUDA graph (DDIM, PLMS, DDPM, LMS, Euler or Euler-ancestral +
classifier-free guidance).

Reference call sites: the loop inside `pipeline(...)` -- inference.py:175-176, 342-351; finetune_sd.py:264-271 -- i.e. per
step `latent_model_input = cat([latents] * 2)`, `unet(...)`, `noise_pred_uncond + guidance_scale * (...)`, `scheduler.step`.

What the graph holds (nothing is launched eagerly between two steps, the host only calls cudaGraphLaunch):

    sampler_advance            in_t <- timesteps[cursor]; cursor += 1            (device-side step index)
    UNet plan                  over the CFG batch [uncond | cond], one launch chain
    cfg_ancestral_step_table   latents <- c_x0 x0 + c_x x + c_e eps (+ c_z z), eps = eps_u + g (eps_c - eps_u), coefficients and
                               the noise row = table[cursor], in place.  DDIMScheduler (eta = 0: no noise rows; eta > 0) and
                               DDPMScheduler.  The noise of every stochastic step sits in a device table that `draw_noise` fills
                               from the caller's generator before the run, outside the graph, in the order the per-call loop
                               draws it.  It holds n_noisy_steps * B*4*h*w floats: 3.3 MB per image at 50 steps and 64x64
                               latents, 2.1 GB for 1000 DDPM steps at batch 32.
    (PNDMScheduler / PLMS: cfg_plms_step_table -- weights, eps-ring slots and the saved-sample flags of this call = table[cursor];
     the 4-deep eps history is a device ring, PNDM's repeated first timestep reads the sample saved by the first call)
    (LMS / Euler / Euler-ancestral: sampler_scale_input replaces the two latents copies -- x2 = [latents | latents] / in_div, the
     model-input scaling of the sigma-space schedulers -- and cfg_sigma_step_table closes the step: sigma, the update weights,
     the LMS derivative-ring slots, the noise row and sigma_up = table[cursor].  The 4-slot derivative ring exists for LMS only,
     the noise table (one row per step, the last one included) for Euler-ancestral only.)
    inpaint_blend_table        inpaint mode only: latents <- m (sa[t] x0 + sb[t] z) + (1 - m) latents at t = timesteps[cursor],
                               the masking step of legacy inpainting; x0, z and m are buffers `run(blend=...)` fills
    (9-channel inpainting UNet (in_channels = out_channels + 5): sampler_inpaint_input replaces the two latents copies and
     sampler_scale_input -- x2 = [latents | cond | latents | cond] (/ in_div for the sigma-space schedulers), the UNet input of
     diffusers 0.7.2's StableDiffusionInpaintPipeline, concatenated before it is scaled.  cond = [mask | masked-image latents]
     (B, 5, h, w) is a buffer `run(cond=...)` fills; the latents, the step and every scheduler buffer keep out_channels.)

A run that starts partway through the schedule (img2img, inpainting: `start` = t_start) holds only the executed steps in its
timestep, coefficient and noise tables, so its graph is launch for launch the text-to-image graph.

`host_step()` is the same graph with the host on both ends: H2D memcpy nodes for the latents and the text context out of
pinned host buffers, the context K/V projections (the context may change every call), the step, and a D2H memcpy node of
the new latents -- what bench.py reports as `e2e`.
"""
from __future__ import annotations

import torch

from . import ops
from ._lib import B200SDError
from .engine import Engine
from .plan import run_plan


class CapturedSampler:
    def __init__(self, unet, scheduler, batch_images, h, w, S_ctx=77, guidance_scale=7.5, lanes=None, eta=0.0, start=0,
                 inpaint=False):
        if not hasattr(scheduler, "captured_step"):
            raise B200SDError("CapturedSampler covers the schedulers of b200sd.schedulers: DDIMScheduler, PNDMScheduler (PLMS), "
                              "DDPMScheduler, LMSDiscreteScheduler, EulerDiscreteScheduler and EulerAncestralDiscreteScheduler")
        if lanes not in (None, 1):
            raise ValueError(f"lanes={lanes}: the step runs the CFG batch as one launch chain.  Concurrent per-half chains were "
                             "slower at every batch size measured (profiles/r02b_lanes_sweep.txt) and were removed")
        plan = scheduler.captured_step(eta, start, inpaint)     # eta reaches only DDIM, as in diffusers' pipeline
        cfg = unet.config
        self.n_cond = cfg.in_channels - cfg.out_channels     # 5 for the inpainting UNet: mask | masked-image latents
        if self.n_cond not in (0, 5):
            raise ValueError(f"a UNet with in_channels={cfg.in_channels}, out_channels={cfg.out_channels} is neither a text-to-image "
                             "nor an inpainting UNet")
        if self.n_cond and (start != 0 or inpaint):
            raise ValueError("the 9-channel inpainting UNet runs the full schedule from noise: start != 0 and the legacy "
                             "masking step (inpaint=True) do not apply to it")
        if unet._precision != "bf16":
            raise B200SDError("CapturedSampler runs the bf16 plan")
        B = int(batch_images)
        self.unet, self.scheduler, self.B, self.h, self.w, self.S, self.lanes = unet, scheduler, B, h, w, S_ctx, 1
        self.guidance = float(guidance_scale)
        dev = self.device = unet.device
        unet._ensure_packed()
        self._pack_gen = unet._pack_gen
        f32 = dict(dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            self.latents = torch.zeros(B, cfg.out_channels, h, w, **f32)       # updated in place by every step
            self.x2 = torch.zeros(2 * B, cfg.in_channels, h, w, **f32)         # [latents | latents] (+ cond), the UNet's input
            self.cond = torch.zeros(B, self.n_cond, h, w, **f32) if self.n_cond else None   # [mask | masked-image latents]
            self.eps = torch.zeros(2 * B, cfg.out_channels, h, w, **f32)       # [uncond | cond] noise predictions
            self.in_t = torch.zeros(2 * B, **f32)
            self.ctx = torch.zeros(2 * B, S_ctx, cfg.cross_attention_dim, **f32)
            ts = [float(t) for t in scheduler.timesteps.tolist()[start:]]
            if not ts:
                raise ValueError(f"start={start} leaves no step of the {len(scheduler.timesteps)}-step schedule")
            self.n_steps = len(ts)
            self.t_table = torch.tensor(ts, **f32)
            self.coef_table = torch.tensor(plan.rows, **f32).contiguous()         # one row per step
            self.noise = torch.zeros(plan.n_noise, self.latents.numel(), **f32)
            self.ring = torch.zeros(plan.ring_slots, self.latents.numel(), **f32)
            self.saved = torch.zeros_like(self.latents) if "saved" in plan.buffers else None
            self._scale_input, self._step = plan.scale_input, plan.step
            self._step_buffers = tuple(getattr(self, b) for b in plan.buffers)
            self.inpaint = bool(inpaint)
            if self.inpaint:         # the init latents before noising, the init noise and the keep-mask, latents-shaped
                self.init_orig, self.blend_noise, self.mask = (torch.zeros_like(self.latents) for _ in range(3))
                self.noise_tables = scheduler._noise_tables(dev)
            self.cursor = torch.zeros(2, dtype=torch.int32, device=dev)
            self.stream = torch.cuda.Stream(device=dev)
            # built under the capture stream: the split-K workspace of the GEMMs is per (device, stream)
            with torch.cuda.stream(self.stream):
                self.engines = [Engine(unet, 2 * B, h, w, S_ctx, dev, io=(self.x2, self.in_t, self.eps))]
            self.graph = None
            self.host_graph = None
            self.kernels_per_step = 0
            self._ctx_key = None

    # -- building blocks ----------------------------------------------------------------------------
    def _project_context(self):
        eng = self.engines[0]
        eng.in_ctx.copy_(self.ctx.reshape(-1, self.ctx.shape[-1]))
        run_plan(eng.ctx_plan)

    def _step_ops(self):
        ops.sampler_advance(self.t_table, self.cursor, self.in_t)
        B = self.B
        if self.n_cond:
            table = (self.coef_table, self.cursor) if self._scale_input else (None, None)
            ops.sampler_inpaint_input(self.latents, self.cond, self.x2, *table)
        elif self._scale_input:
            ops.sampler_scale_input(self.latents, self.x2, self.coef_table, self.cursor)
        else:
            self.x2[:B].copy_(self.latents)
            self.x2[B:].copy_(self.latents)
        run_plan(self.engines[0].plan)
        self._step(self.eps[:B], self.eps[B:], self.latents, *self._step_buffers, self.guidance, self.coef_table, self.cursor)
        if self.inpaint:
            ops.inpaint_blend_table(self.latents, self.init_orig, self.blend_noise, self.mask, self.t_table, self.cursor,
                                    *self.noise_tables)

    def _capture(self, body):
        """Warm up `body` on the capture stream (lazy one-time setup: function attributes, per-stream workspaces), then capture."""
        s0 = self.stream
        s0.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s0):
            body()
        s0.synchronize()
        cur = int(self.cursor[0])      # the warm-up advanced the device-side step index: put it back
        self.cursor[0] = (cur - 1) % self.n_steps
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        before = ops.launch_count()
        with torch.cuda.graph(g, stream=s0):
            body()
        return g, ops.launch_count() - before

    # -- public surface -----------------------------------------------------------------------------
    def reset(self, step=0):
        """the next step() executes scheduler.timesteps[start + step]"""
        self.cursor.copy_(torch.tensor([step % self.n_steps, 0], dtype=torch.int32))

    def set_context(self, ctx2):
        """ctx2 = cat([uncond, cond]) (2B, S, 768): projected once to every cross-attention's K/V"""
        if tuple(ctx2.shape) != tuple(self.ctx.shape):
            raise ValueError(f"encoder_hidden_states must be {tuple(self.ctx.shape)}, got {tuple(ctx2.shape)}")
        with torch.cuda.device(self.device):
            self.ctx.copy_(ctx2)
            self._project_context()

    def set_latents(self, latents):
        self.latents.copy_(latents)

    def step(self):
        """one denoising iteration: ONE cudaGraphLaunch, no eager kernels"""
        with torch.cuda.device(self.device):
            if self.graph is None:
                keep = self.latents.clone()
                self.graph, self.kernels_per_step = self._capture(self._step_ops)
                self.latents.copy_(keep)       # the warm-up run updated the latents in place
            self.graph.replay()

    def draw_noise(self, generator=None):
        """Fill the noise table: one schedulers.step_noise draw per stochastic step, in step order -- the same numbers the
        per-call loop draws from the same generator.  DDIM with eta = 0, PLMS, LMS and Euler draw nothing."""
        from .schedulers import step_noise
        with torch.cuda.device(self.device):
            for k in range(self.noise.shape[0]):
                step_noise(self.latents, generator, out=self.noise[k].view(self.latents.shape))

    def set_blend(self, init_orig, noise, mask):
        """inpaint mode: the init latents before noising, the init noise (both (B,4,h,w)) and the keep-mask (broadcastable to
        them; 1 = keep) that every step's blend reads"""
        if not self.inpaint:
            raise ValueError("this sampler was built without inpaint=True")
        for buf, t in ((self.init_orig, init_orig), (self.blend_noise, noise), (self.mask, mask)):
            buf.copy_(t.float().expand_as(buf))

    def set_cond(self, mask, masked_latents):
        """9-channel UNet: the mask (B or 1, 1, h, w) and the masked-image latents (B or 1, 4, h, w) that every step's UNet input
        carries after the latents"""
        if not self.n_cond:
            raise ValueError("cond=(mask, masked_latents) is for a 9-channel inpainting UNet")
        B, h, w = self.B, self.h, self.w
        if tuple(mask.shape[1:]) != (1, h, w) or tuple(masked_latents.shape[1:]) != (self.n_cond - 1, h, w):
            raise ValueError(f"cond: mask must be (B, 1, {h}, {w}) and masked_latents (B, {self.n_cond - 1}, {h}, {w}), got "
                             f"{tuple(mask.shape)} and {tuple(masked_latents.shape)}")
        self.cond[:, :1].copy_(mask.float().expand(B, 1, h, w))
        self.cond[:, 1:].copy_(masked_latents.float().expand(B, self.n_cond - 1, h, w))

    @torch.no_grad()
    def run(self, latents, ctx2, generator=None, blend=None, cond=None):
        """latents (B,4,h,w) -> denoised latents after the steps timesteps[start:].  A stochastic sampler first draws its step
        noise from `generator` (draw_noise).  An inpainting sampler needs blend=(init_orig, noise, mask) (set_blend), a 9-channel
        UNet cond=(mask, masked_latents) (set_cond)."""
        if self.unet._stale(self._pack_gen):
            raise B200SDError("the UNet's weights changed after this sampler was built: build a new CapturedSampler")
        if (blend is not None) != self.inpaint:
            raise ValueError("blend=(init_orig, noise, mask) is required in inpaint mode and only there")
        if (cond is not None) != bool(self.n_cond):
            raise ValueError("cond=(mask, masked_latents) is required with a 9-channel inpainting UNet and only there")
        if blend is not None:
            self.set_blend(*blend)
        if cond is not None:
            self.set_cond(*cond)
        self.set_context(ctx2.float())
        self.set_latents(latents.float() * self.scheduler.init_noise_sigma)
        self.draw_noise(generator)
        self.reset(0)
        for _ in range(self.n_steps):
            self.step()
        return self.latents.clone()

    def bind_host(self, lat_host, ctx_host, out_host):
        """Capture the host-facing step over these PINNED host buffers (latents in, context in, new latents out)."""
        for t in (lat_host, ctx_host, out_host):
            if not t.is_pinned():
                raise B200SDError("host_step needs pinned host buffers")

        def body():
            self.latents.copy_(lat_host, non_blocking=True)
            self.ctx.copy_(ctx_host, non_blocking=True)
            self._project_context()
            self._step_ops()
            out_host.copy_(self.latents, non_blocking=True)
        with torch.cuda.device(self.device):
            self.host_graph, self.kernels_per_host_step = self._capture(body)
        self._host = (lat_host, ctx_host, out_host)

    def host_step(self):
        """H2D(latents, context) -> context K/V -> step -> D2H(latents): one graph launch + one stream synchronize"""
        with torch.cuda.device(self.device):
            self.host_graph.replay()
            torch.cuda.current_stream().synchronize()
