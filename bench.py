#!/usr/bin/env python
"""bench.py -- SD v1.5 UNet denoise hot path on B200 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one denoising iteration of the 50-step DDIM + classifier-free-guidance sampler for B
images per GPU at 512x512: x2 = cat([lat, lat]) -> UNet(2B,4,64,64; t; ctx (2B,77,768)) ->
fused CFG combine + DDIM update.  Metric: denoising iterations per second (whole job, all GPUs);
images/s = it/s / 50 is reported next to it.  Sampling shards by image with no collective
("scaling": "weak": every GPU runs its own B images).

Output: ONE JSON line (see README / DESIGN.md section "Measurement").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_SAMPLE_64 = 0.8033e12  # SURVEY.md App. C: UNet fwd per sample @ 64x64 latent, 2*MAC


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# stdout carries the JSON line(s) of this script and NOTHING else: the process that does the work moves file descriptor 1 onto
# stderr (C-level writers included -- NCCL prints its "NCCL version ..." banner to stdout from inside init_process_group) and
# writes its result lines to a private duplicate of the original stdout.
# ---------------------------------------------------------------------------------------------------
_RESULT_OUT = None


def _claim_stdout():
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(text):
    if _RESULT_OUT is None:
        print(text, flush=True)
    else:
        _RESULT_OUT.write(text + "\n")
        _RESULT_OUT.flush()



def ddim_coefs(sch, t):
    return sch._coefs(t)


def sample_config(batch, world, total_images, portrait):
    """`config` of the sampling workload -- ONE builder for our arm and the reference arm, so that the two lines name the
    workload identically (the driver compares the dicts)."""
    h, w = (96, 64) if portrait else (64, 64)
    return {"workload": "sd15_unet_ddim50_cfg7.5_" + ("512x768" if portrait else "512px"),
            "images_per_gpu": batch, "total_images": total_images if total_images > 0 else batch * world,
            "unet_batch": 2 * batch, "latent": f"4x{h}x{w}", "context": "77x768",
            "weights": "random-init SD v1.5 UNet (859.5M params)", "guidance_scale": 7.5, "scheduler": "DDIM, 50 steps"}


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the fp32 oracle (restated diffusers 0.7.2 math) on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_oracle_it_per_s(batch_images, budget_s, max_iters, warmup=1, hw=(64, 64)):
    import torch
    from oracle.unet_ref import make_oracle_unet
    from oracle import schedulers_ref as R
    torch.set_num_threads(os.cpu_count() or 1)
    m = make_oracle_unet(seed=0)
    sch = R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False)
    sch.set_timesteps(50)
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(batch_images, 4, hw[0], hw[1], generator=g)
    ctx2 = torch.randn(2 * batch_images, 77, 768, generator=g)
    ts = sch.timesteps.tolist()
    done, t_total = 0, 0.0
    with torch.no_grad():
        for i in range(warmup + max_iters):
            t = ts[i % len(ts)]
            t0 = time.perf_counter()
            eps = m(torch.cat([lat] * 2), t, ctx2).sample
            eps = R.cfg_combine(eps, 7.5)
            lat = sch.step(eps, t, lat).prev_sample
            dt = time.perf_counter() - t0
            if i >= warmup:
                done += 1
                t_total += dt
                if t_total > budget_s:
                    break
    return done * batch_images / t_total, done, t_total, torch.get_num_threads()


def run_reference(args):
    _claim_stdout()
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    v, done, t_total, cores = cpu_oracle_it_per_s(args.batch, budget_s=150.0, max_iters=args.steps, warmup=min(args.warmup, 1),
                                                  hw=(96, 64) if args.portrait else (64, 64))
    sample = f"{done} of {args.steps} denoising iterations (time-bounded), fp32 oracle on host CPU, CFG batch {2 * args.batch}"
    line = {
        "impl": "reference", "metric": "unet_denoise_it_per_s", "value": v, "unit": "it/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(done, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": sample_config(args.batch, args.gpus, args.total_images, args.portrait), "images_per_s": v / 50.0,
        "cpu_baseline": {"value": v, "unit": "it/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# library bar (SURVEY.md 8(d) "extra comparator"): the oracle module itself on the GPU in bf16 under eager torch
# (cuDNN / cuBLASLt kernels), attention as the reference's diffusers materialises it and again through torch SDPA.
# Not the reference arm and not part of the driver contract -- a reported yardstick for the same workload.
# ---------------------------------------------------------------------------------------------------
def run_library(args):
    _claim_stdout()
    if int(os.environ.get("RANK", 0)) != 0:
        return
    import torch
    import torch.nn.functional as F
    from oracle import unet_ref
    dev = torch.device("cuda", 0)
    B = args.batch
    h, w = (96, 64) if args.portrait else (64, 64)
    m = unet_ref.make_oracle_unet(seed=0).to(dev).bfloat16().eval()
    g = torch.Generator().manual_seed(42)
    x = torch.randn(2 * B, 4, h, w, generator=g).to(dev).bfloat16()
    ctx = torch.randn(2 * B, 77, 768, generator=g).to(dev).bfloat16()

    def timed():
        with torch.no_grad():
            for _ in range(max(args.warmup, 3)):
                m(x, 500, ctx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.steps):
                m(x, 980 - 20 * (i % 50), ctx)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    ms_mat = timed()

    def sdpa_forward(self, xx, context=None):
        context = xx if context is None else context
        b, s, c = xx.shape
        hh = self.heads
        q = self.to_q(xx).view(b, s, hh, c // hh).transpose(1, 2)
        k = self.to_k(context).view(b, -1, hh, c // hh).transpose(1, 2)
        v = self.to_v(context).view(b, -1, hh, c // hh).transpose(1, 2)
        o = F.scaled_dot_product_attention(q, k, v, scale=self.scale).transpose(1, 2).reshape(b, s, c)
        return self.to_out[0](o)

    orig = unet_ref.CrossAttention.forward
    unet_ref.CrossAttention.forward = sdpa_forward
    try:
        ms_sdpa = timed()
    finally:
        unet_ref.CrossAttention.forward = orig
    best = min(ms_mat, ms_sdpa)
    emit(json.dumps({
        "impl": "library", "metric": "unet_denoise_it_per_s", "value": B * 1e3 / best, "unit": "it/s", "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": best, "higher_is_better": True, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "sd15_unet_cfg_batch%d_%s" % (2 * B, "512x768" if args.portrait else "512px"),
                   "what": "fp32-oracle module .cuda().bfloat16() under eager torch %s (cuDNN/cuBLASLt), UNet call only" % torch.__version__,
                   "ms_per_step_materialised_attention": ms_mat, "ms_per_step_sdpa_attention": ms_sdpa}}))


def shard_images(total: int, world: int, rank: int) -> int:
    """SURVEY.md 8(e): images of one batch are independent units -- contiguous chunks, remainder to the low ranks; a rank
    may get none (B < #GPUs)."""
    return total // world + (1 if rank < total % world else 0)


# ---------------------------------------------------------------------------------------------------
# elementwise kernels (north_star subsystem 3): achieved HBM GB/s, SURVEY.md 8(d) algorithmic bytes
# ---------------------------------------------------------------------------------------------------
def elementwise_gbs(dev):
    """cfg_ddim_step / cfg_plms_step / add_noise / mse at the REAL size of the workload (one 4x64x64 latent: 16 384 elements --
    launch-latency-bound, a few hundred KB moved) and at a saturating 64 Mi elements (every operand larger than the 126 MB L2,
    so each launch streams from HBM).  fp32 operands.  Each kernel: 3 warm-up launches, then `reps` launches captured into one
    CUDA graph, CUDA-event timed.  bytes = operands the kernel must read + results it must write (stated per kernel)."""
    import torch
    from b200sd import ops
    hbm, _, _, which = _peaks()
    out = {"peak_gbs": hbm, "peak_kind": f"HBM copy bandwidth, {which}", "dtype": "f32", "sizes": {}}
    sa = torch.linspace(0.99, 0.07, 1000, device=dev)
    sb = (1 - sa * sa).sqrt()

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        with torch.cuda.graph(g, stream=side):
            for _ in range(reps):
                fn()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    for label, B, E1, reps in (("real_1x4x64x64", 1, 4 * 64 * 64, 50), ("saturating_64Mi", 64, 1 << 20, 5)):
        E = B * E1
        mk = lambda: torch.randn(B, E1, device=dev)
        eu, ec, x, o, eo, h1, h2, h3 = (mk() for _ in range(8))
        t = torch.randint(0, 1000, (B,), device=dev)
        rec = {}
        cases = {
            # name: (callable, bytes moved, formula)
            "cfg_ddim_step": (lambda: ops.cfg_ddim_step(eu, ec, x, 7.5, 0.9, 0.43, 0.92, 0.39, out=o), 4 * E * 4,
                              "4*E*b: read eps_u, eps_c, x; write x'"),
            "cfg_plms_step": (lambda: ops.cfg_plms_step(eu, ec, x, [h1, h2, h3], [55 / 24, -59 / 24, 37 / 24, -9 / 24], 7.5, 1.01, 0.02,
                                                        out=o, eps_out=eo), 8 * E * 4,
                              "(k+5)*E*b, k=3: read eps_u, eps_c, x, 3 history eps; write x', combined eps (history)"),
            "add_noise": (lambda: ops.add_noise(x, eu, t, sa, sb, out=o), 3 * E * 4, "3*E*b: read x0, noise; write x_t (+8 B/sample)"),
            "mse_loss_fwd": (lambda: ops.mse_loss_fwd(eu, ec), 2 * E * 4, "2*E*b: read pred, target"),
        }
        if label.startswith("saturating"):
            # the optimizer step of the fine-tuning path (SURVEY.md 8f N2; finetune_sd.py:407-420, 569): fp32-moment AdamW and the
            # reference's default, block-wise 8-bit AdamW, over E parameters of a flat buffer (fused: gradient scaling, bf16
            # re-cast of the weights, gradient zeroing)
            from b200sd.trainer import create_dynamic_map
            pf, gf = eu.view(-1), ec.view(-1).mul_(0.01)
            mf, vf = torch.zeros(E, device=dev), torch.zeros(E, device=dev)
            wbf = torch.empty(E, device=dev, dtype=torch.bfloat16)
            c1, c2 = torch.zeros(E, device=dev, dtype=torch.uint8), torch.zeros(E, device=dev, dtype=torch.uint8)
            am1, am2 = torch.zeros(E // 2048, device=dev), torch.zeros(E // 2048, device=dev)
            q1, q2 = create_dynamic_map(True).to(dev), create_dynamic_map(False).to(dev)
            cases["adamw_step"] = (lambda: ops.adamw_step(pf, gf, mf, vf, wbf, 1e-5, 0.9, 0.999, 1e-8, 1e-2, 1, grad_scale=1.0,
                                                          zero_grad=True), 34 * E,
                                   "34 B/param: read p, g, m, v (fp32); write p, m, v, zeroed g (fp32) + bf16 weights")
            cases["adamw8bit_step"] = (lambda: ops.adamw8bit_step(pf, gf, c1, c2, am1, am2, q1, q2, None, None, None, wbf, 1e-5, 0.9,
                                                                  0.999, 1e-8, 1e-2, 1, grad_scale=1.0, zero_grad=True), 22 * E,
                                       "22 B/param: read p, g (fp32) + 2 moment codes (u8); write p, zeroed g (fp32), bf16 weights, 2 codes")
        for name, (fn, nbytes, formula) in cases.items():
            sec = timed(fn, reps)
            rec[name] = {"us": round(sec * 1e6, 2), "bytes": nbytes, "gbs": round(nbytes / sec / 1e9, 1),
                         "frac_of_hbm_peak": round(nbytes / sec / 1e9 / hbm, 4), "bytes_formula": formula}
        out["sizes"][label] = {"elements": E, "kernels": rec}
    return out


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
class _PerCallSampler:
    """The per-call loop of pipeline.denoise_loop behind CapturedSampler's surface (fp32-accuracy plan; PLMS)."""

    def __init__(self, unet, sch, B, h, w, dev):
        import torch
        self.unet, self.sch, self.B = unet, sch, B
        self.ts = sch.timesteps.tolist()
        self.i = 0
        self.x2 = torch.empty(2 * B, 4, h, w, device=dev)
        self.latents = torch.empty(B, 4, h, w, device=dev)
        self.nxt = torch.empty_like(self.latents)
        self.ctx = None
        self.kernels_per_step = 0
        self.lanes = 1

    def set_context(self, ctx):
        self.ctx = ctx

    def set_latents(self, lat):
        self.latents.copy_(lat)

    def reset(self, step=0):
        self.i = step

    def step(self):
        t = self.ts[self.i % len(self.ts)]
        self.i += 1
        B = self.B
        self.x2[:B].copy_(self.latents)
        self.x2[B:].copy_(self.latents)
        eps2 = self.eps = self.unet(self.x2, t, self.ctx).sample
        self.sch.step_cfg(eps2, t, self.latents, 7.5, out=self.nxt)
        self.latents, self.nxt = self.nxt, self.latents
        eng = next(iter(self.unet._engines.values()))
        self.kernels_per_step = getattr(eng, "kernels_per_graph", 0)
        self.engines = [eng]

    def bind_host(self, lat_host, ctx_host, out_host):
        import torch
        self._host = (lat_host, ctx_host, out_host)
        self._ctx_d = torch.empty_like(ctx_host, device=self.latents.device)

    def host_step(self):
        import torch
        lat_host, ctx_host, out_host = self._host
        self.latents.copy_(lat_host, non_blocking=True)
        self._ctx_d.copy_(ctx_host, non_blocking=True)
        self.ctx = self._ctx_d
        self.step()
        out_host.copy_(self.latents, non_blocking=True)
        torch.cuda.current_stream().synchronize()


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, tensors):
    """Write each tensor as out_dir/<name>.npy in float32, so that two builds run with the same arguments can be compared output
    for output.  When the tensors hold more than DUMP_BYTES together, each is replaced by the same seeded sample of its flattened
    elements (ascending indices), sized so that the files stay within DUMP_BYTES."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.size * (DUMP_BYTES - 256 * len(arrays)) // total          # 256: room for each .npy header
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    _claim_stdout()
    import torch
    import torch.distributed as dist
    from b200sd import ops
    from b200sd.schedulers import DDIMScheduler
    from b200sd.unet import UNet2DConditionModel

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    if args.total_images > 0:
        # BASELINE config 5: a fixed batch of images sharded over the GPUs (contiguous chunks, remainder to the low ranks;
        # ranks left without an image idle) -> strong scaling, no collective on the data path
        B = shard_images(args.total_images, world, rank)
    idle = B == 0
    if idle:
        B = 1          # keeps the buffers valid; this rank runs no steps and contributes no images
    h, w = (96, 64) if args.portrait else (64, 64)
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(dev).eval()          # random-init weights of the SD v1.5 architecture
    if args.precision == "fp32":
        unet.set_precision("fp32")
    sch = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                        set_alpha_to_one=False)
    sch.set_timesteps(50)
    ts = sch.timesteps.tolist()
    g = torch.Generator().manual_seed(42 + rank)
    lat_host = torch.randn(B, 4, h, w, generator=g).pin_memory()
    ctx_host = torch.randn(2 * B, 77, 768, generator=g).pin_memory()
    lat = lat_host.to(dev)
    ctx = ctx_host.to(dev)
    # The step a user runs: b200sd.sampler.CapturedSampler -- timestep, UNet plan (one launch chain per CFG half = "lane"), CFG
    # combine + DDIM update as ONE CUDA graph; pipeline.denoise_loop uses the same object.  --lanes 0 = the library's default.
    # (--precision fp32, the accuracy path, keeps the per-call loop: UNet graph + one eager CFG/DDIM kernel per step.)
    from b200sd.sampler import CapturedSampler
    smp = CapturedSampler(unet, sch, B, h, w, 77, 7.5, lanes=(args.lanes or None)) if args.precision == "bf16" else _PerCallSampler(unet, sch, B, h, w, dev)

    def step(i):
        smp.step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        smp.set_context(ctx)
        smp.set_latents(lat)
        smp.reset(0)
        for i in range(max(args.warmup, 3)):
            step(i)          # idle ranks warm up too (keeps the code path uniform), but run no timed steps
        eng = smp.engines[0]
        # ---- device-resident timing ----
        barrier()
        sampler = ClockSampler(local) if rank == 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = ops.launch_count()
        e0.record()
        for i in range(0 if idle else args.steps):
            step(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        eager_launches = ops.launch_count() - launches0
        gpu_launches = eager_launches + smp.kernels_per_step * (0 if idle else args.steps)
        if args.dump_outputs and rank == 0:
            # the step below (end to end) keeps updating the same buffers: keep what the last timed step returned
            dump_outputs(args.dump_outputs, {"latents": smp.latents, "noise_pred": smp.eps})

        # ---- end to end through the public API with host buffers (H2D + D2H inside the timed region): every step copies the
        # latents and the text context out of pinned host memory, projects the context, runs the step and copies the new
        # latents back; the host waits for them and feeds them to the next step ----
        out_host = torch.empty(B, 4, h, w).pin_memory()
        smp.bind_host(lat_host, ctx_host, out_host)

        def e2e_step(i):
            smp.host_step()
            lat_host.copy_(out_host)

        for i in range(3):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(0 if idle else args.steps):
            e2e_step(i)
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        clocks = sampler.stop() if sampler else None      # sampled over both timed regions (device-resident + end to end)

        images_total = (0 if idle else B) * 1.0
        if world > 1:
            tt = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms, e2e_ms = float(tt[0]), float(tt[1])
            ti = torch.tensor([images_total], device=dev, dtype=torch.float64)
            dist.all_reduce(ti, op=dist.ReduceOp.SUM)
            images_total = float(ti[0])

        # ---- roofline of the dominant kernel (tcgen05 GEMM / implicit-GEMM conv), timed live INSIDE the captured step ----
        roof = None
        kernels = None
        if rank == 0 and args.precision == "bf16" and not idle:
            acc, per_op, instrumented_ms = eng.profile(iters=5)
            hbm, tf_burst, tf_sus, which = _peaks()
            mm_ms = sum(acc[k][0] for k in ("gemm", "conv3x3") if k in acc)
            mm_fl = sum(acc[k][1] for k in ("gemm", "conv3x3") if k in acc)
            mm_n = sum(acc[k][2] for k in ("gemm", "conv3x3") if k in acc)
            # `eng` is the plan of ONE lane (its share of the CFG batch); the step runs smp.lanes such chains side by side, so
            # the step's FLOPs and launches are lanes x the lane's, and the kernel's share of a lane's chain is its share of
            # the step
            mm_fl *= smp.lanes
            mm_n *= smp.lanes
            # The event-record nodes serialise the graph (no tail / launch overlap between kernels) and stretch every interval
            # by a few us: the kernel's SHARE of the instrumented step is what carries over, so its time inside the real step
            # is share x the un-instrumented step time measured above.
            share = mm_ms / max(instrumented_ms, 1e-9)
            step_ms = ms / max(args.steps, 1)
            mm_ms_in_step = share * step_ms
            achieved = mm_fl / (mm_ms_in_step * 1e-3) / 1e12 if mm_ms_in_step > 0 else 0.0
            traffic = None
            for tp in ("r02_traffic.json", "r01_traffic.json"):
                tp = os.path.join(ROOT, "profiles", tp)
                if os.path.exists(tp) and B == 1 and not args.portrait:
                    with open(tp) as f:
                        traffic = json.load(f)["gemm_tcgen05_kernel"]["dram_bytes_per_launch"]   # ncu, per launch, same workload
                    break
            # the kernel is timed inside a long step -> the SUSTAINED bf16 peak is the denominator; the burst fraction is
            # printed next to it
            roof = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (GEMM + implicit-GEMM conv3x3)",
                    "achieved": achieved, "peak": tf_sus, "unit": "TFLOP/s", "frac": achieved / tf_sus,
                    "peak_kind": f"bf16 sustained, {which}", "frac_of_burst_peak": achieved / tf_burst, "burst_peak": tf_burst,
                    "launches_per_step": mm_n, "avg_launch_us": 1e3 * mm_ms_in_step / max(mm_n, 1), "flops_per_step": mm_fl,
                    "share_of_step": share, "avg_launch_us_instrumented": 1e3 * mm_ms / max(mm_n, 1),
                    "how": "CUDA-graph replay of the step with an event-record node between consecutive kernels (cold weights "
                           "from HBM, true predecessor in L2) gives the kernel's share of the step; achieved = FLOPs / "
                           "(share x un-instrumented ms_per_step)" + (f"; the step runs {smp.lanes} independent launch chains "
                           "(one per CFG half) concurrently: share is measured on one chain, FLOPs and launches count all of them" if smp.lanes > 1 else ""),
                    "traffic": traffic,
                    "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)"}
            tot = sum(v[0] for v in acc.values())
            kernels = {k: {"ms_per_step": round(v[0], 4), "share": round(v[0] / tot, 4), "launches": v[2],
                           "tflops": round(v[1] / (v[0] * 1e-3) / 1e12, 1) if v[1] > 0 and v[0] > 0 else None}
                       for k, v in sorted(acc.items(), key=lambda kv: -kv[1][0])}
            kernels["_instrumented_step_ms"] = round(instrumented_ms, 4)
            if args.dump_ops:
                with open(args.dump_ops, "w") as f:
                    f.write(f"# {len(per_op)} launches, in-step (instrumented graph replay {instrumented_ms:.3f} ms)\n")
                    for name, t_ms, fl in sorted(per_op, key=lambda r: -r[1]):
                        f.write(f"{t_ms * 1e3:9.1f} us  {fl / (t_ms * 1e-3) / 1e12 if fl else 0:8.1f} TF/s  {name}\n")

    elementwise = None
    if rank == 0 and args.precision == "bf16" and not args.no_elementwise:
        elementwise = elementwise_gbs(dev)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, done, t_total, cores = cpu_oracle_it_per_s(B, budget_s=20.0, max_iters=3, warmup=1)
        cpu = {"value": v, "unit": "it/s", "cores": cores, "kind": "port",
               "sample": f"{done} denoising iterations (CFG batch {2 * B}, fp32 oracle, 1 warm-up) in {t_total:.1f} s"}

    if rank == 0:
        its = (images_total if args.total_images > 0 else B * world) * args.steps
        value = its / (ms * 1e-3)
        e2e_value = its / (e2e_ms * 1e-3)
        flops_per_it = 2 * (1.2953e12 if args.portrait else FLOPS_PER_SAMPLE_64)
        line = {
            "metric": "unet_denoise_it_per_s", "value": value, "unit": "it/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.total_images > 0 else "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32 (split-bf16 3-term products on the tensor cores)",
            "data": "synthetic",
            "config": sample_config(args.batch if args.total_images <= 0 else B, world, args.total_images, args.portrait),
            "images_per_s": value / 50.0, "e2e_images_per_s": e2e_value / 50.0, "tflops_end_to_end": value * flops_per_it / 1e12,
            "lanes": smp.lanes,
            "l2": "no flush: the 1.72 GB of bf16 weights streamed every step exceed the 126 MB L2", "cuda_graph": True,
            "e2e": {"value": e2e_value, "unit": "it/s",
                    "h2d_bytes_per_step": int(lat_host.numel() * 4 + ctx_host.numel() * 4),
                    "d2h_bytes_per_step": int(out_host.numel() * 4)},
            "gpu_launches": int(gpu_launches), "clocks": clocks, "roofline": roof, "kernels": kernels,
            "elementwise": elementwise, "cpu_baseline": cpu,
        }
    # ---- fine-tuning legs (BASELINE configs[2] / [3]) inside the same line: the gradient-allreduce path is the only
    # collective of the hot path, and the driver's scaling run only ever launches `bench.py --gpus N` ----
    train = train_text = t2i = None
    if args.precision == "bf16" and args.total_images <= 0 and not args.portrait and not args.no_train_legs:
        unet._engines = {}                       # the sampling plan's buffers are not needed any more
        del smp, eng, step, e2e_step
        torch.cuda.empty_cache()
        if rank == 0:
            t2i = text_to_image_leg(dev, unet)
            torch.cuda.empty_cache()
        train = train_leg(dev, world, rank, steps=5, warmup=3, unet=unet)          # same model object: one 860 M-parameter init per rank
        torch.cuda.empty_cache()
        train_text = train_text_leg(dev, world, rank, local, steps=5, warmup=3, unet=unet)
    if rank == 0:
        line["text_to_image"] = t2i
        line["train"] = train
        line["train_text"] = train_text
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# BASELINE configs[4]: book-cover portrait (512 x 768) batched generation, batch 1-64 sharded over the GPUs
# ---------------------------------------------------------------------------------------------------
def run_sweep(args):
    """`--workload sweep [--portrait]`: for every total batch B in --sweep-batches, shard the B images over the ranks (contiguous
    chunks, remainder to the low ranks, ranks without an image idle), run `steps` denoising iterations of the 50-step CFG DDIM
    sampler and print ONE JSON line per B: whole-job images/s = B / (50 * max-over-ranks ms per iteration).  One model per rank,
    no collective on the data path."""
    _claim_stdout()
    import torch
    import torch.distributed as dist
    from b200sd.schedulers import DDIMScheduler
    from b200sd.unet import UNet2DConditionModel
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    h, w = (96, 64) if args.portrait else (64, 64)
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(dev).eval()
    sch = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, set_alpha_to_one=False)
    sch.set_timesteps(50)
    ts = sch.timesteps.tolist()
    flops_per_img_it = 2 * (1.2953e12 if args.portrait else FLOPS_PER_SAMPLE_64)
    for total in [int(x) for x in args.sweep_batches.split(",")]:
        B = shard_images(total, world, rank)
        idle = B == 0
        ms = 0.0
        if not idle:
            g = torch.Generator().manual_seed(42 + rank)
            lat = torch.randn(B, 4, h, w, generator=g).to(dev)
            ctx = torch.randn(2 * B, 77, 768, generator=g).to(dev)
            from b200sd.sampler import CapturedSampler
            smp = CapturedSampler(unet, sch, B, h, w, 77, 7.5)       # the whole step as one CUDA graph (what denoise_loop runs)
            smp.set_context(ctx)
            smp.set_latents(lat)
            smp.reset(0)
            with torch.no_grad():
                def step(i):
                    smp.step()
                for i in range(max(args.warmup, 3)):
                    step(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if not idle:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.no_grad():
                e0.record()
                for i in range(args.steps):
                    step(i)
                e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if not idle:
            ms = e0.elapsed_time(e1) / args.steps
        active = torch.tensor([ms, 0.0 if idle else 1.0], device=dev, dtype=torch.float64)
        if world > 1:
            mx = active.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(active, op=dist.ReduceOp.SUM)
            ms_max, n_active = float(mx[0]), int(active[1])
        else:
            ms_max, n_active = ms, 0 if idle else 1
        if rank == 0:
            ips = total / (50.0 * ms_max * 1e-3)
            emit(json.dumps({"metric": "images_per_s", "value": ips, "unit": "images/s", "n_gpus": world, "gpus_active": n_active,
                              "gpus_idle": world - n_active, "total_images": total, "images_on_rank0": B if not idle else 0,
                              "ms_per_iteration_max_over_ranks": ms_max, "steps": args.steps, "scaling": "strong", "dtype": "bf16",
                              "tflops_per_active_gpu": (total / max(n_active, 1)) * flops_per_img_it / (ms_max * 1e-3) / 1e12 if ms_max else 0,
                              "config": sample_config(B, world, total, args.portrait)}))
        unet._engines = {}
        smp = step = None
        torch.cuda.empty_cache()
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# fine-tuning step (BASELINE config 3): add_noise + UNet fwd/bwd + MSE + gradient allreduce + AdamW
# ---------------------------------------------------------------------------------------------------
def cpu_oracle_train_samples_per_s(batch, steps):
    import torch
    import torch.nn.functional as F
    from oracle.unet_ref import make_oracle_unet
    from oracle import schedulers_ref as R
    torch.set_num_threads(os.cpu_count() or 1)
    m = make_oracle_unet(seed=0).train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-5)
    sch = R.DDPMSchedulerRef() if hasattr(R, "DDPMSchedulerRef") else None
    g = torch.Generator().manual_seed(0)
    x0 = torch.randn(batch, 4, 64, 64, generator=g)
    ctx = torch.randn(batch, 77, 768, generator=g)
    t_total, done = 0.0, 0
    for i in range(steps):
        noise = torch.randn(batch, 4, 64, 64, generator=g)
        t = torch.randint(0, 1000, (batch,), generator=g)
        t0 = time.perf_counter()
        noisy = sch.add_noise(x0, noise, t) if sch is not None else x0 + noise
        loss = F.mse_loss(m(noisy, t, ctx).sample, noise)
        loss.backward()
        opt.step()
        opt.zero_grad()
        t_total += time.perf_counter() - t0
        done += 1
    return done * batch / t_total, done, t_total, torch.get_num_threads()


def _timed_steps(step_fn, steps, warmup, world, dev):
    """W untimed + K timed calls of step_fn, barrier + synchronize on both sides, CUDA events, MAX over ranks -> ms/step."""
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        step_fn()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step_fn()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        tt = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt[0])
    return ms


def train_leg(dev, world, rank, steps=5, warmup=3, B=8, unet=None):
    """BASELINE configs[2] inside the default bench line: `steps` UNet fine-tuning steps at batch 8/GPU (add_noise + UNet fwd +
    MSE + bwd + bucketed NCCL allreduce of the 859.5 M fp32 gradients + fused AdamW), then the SAME steps with the collective
    switched off (every rank steps on its local gradient) -- the difference is the exposed (non-overlapped) communication."""
    import torch
    from b200sd.schedulers import DDPMScheduler
    from b200sd.trainer import Trainer
    from b200sd.unet import UNet2DConditionModel
    if unet is None:
        torch.manual_seed(0)
        unet = UNet2DConditionModel().to(dev)          # identical initial weights on every rank
    unet.requires_grad_(True)
    sched = DDPMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    tr = Trainer(unet, sched, lr=1e-5, weight_decay=1e-2)
    g = torch.Generator().manual_seed(1000 + rank)
    x0, noise = torch.randn(B, 4, 64, 64, generator=g).to(dev), torch.randn(B, 4, 64, 64, generator=g).to(dev)
    t, ctx = torch.randint(0, 1000, (B,), generator=g).to(dev), torch.randn(B, 77, 768, generator=g).to(dev)
    step = lambda: tr.train_step(x0, noise, t, ctx)
    ms = _timed_steps(step, steps, warmup, world, dev)
    tr.allreduce_enabled = False
    ms_local = _timed_steps(step, steps, 1, world, dev)
    tr.allreduce_enabled = True
    loss = float(step())
    n_param = sum(p.numel() for p in unet.parameters())
    _, _, tf_sus, _ = _peaks()
    flops_step = 3 * B * FLOPS_PER_SAMPLE_64
    rec = {"workload": "sd15_unet_finetune_512px", "batch_per_gpu": B, "steps": steps, "warmup": warmup, "n_gpus": world,
           "ms_per_step": ms, "samples_per_s": B * world / (ms * 1e-3), "ms_per_step_without_allreduce": ms_local,
           "exposed_comm_ms": ms - ms_local, "allreduce_bytes_on_wire_per_gpu": int(2 * (world - 1) / world * n_param * 4),
           "tflops_per_gpu": flops_step / (ms * 1e-3) / 1e12, "frac_of_sustained_bf16_peak": flops_step / (ms * 1e-3) / 1e12 / tf_sus,
           "last_loss": loss, "collective": "NCCL all_reduce(SUM) of the flat fp32 gradient buffer in 64 MB buckets, overlapped with the backward"}
    del tr
    return rec


def text_to_image_leg(dev, unet, images=(1, 4), reps=3):
    """The whole `pipeline(prompt_ids, 512, 512, 50 steps, CFG 7.5)` call of inference.py:175-176, 342-351 on b200sd's own
    models: CLIP text encoder over the [uncond | cond] token ids -> 50 captured DDIM steps -> VAE decode -> uint8 image on the
    host.  Random-init SD v1.x architectures, synthetic token ids; H2D of the ids and D2H of the images inside the timed region."""
    import torch
    from b200sd.clip import CLIPTextModel
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    from b200sd.vae import AutoencoderKL
    torch.manual_seed(0)
    clip = CLIPTextModel().to(dev).eval().requires_grad_(False)
    vae = AutoencoderKL().to(dev).eval()
    sch = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, set_alpha_to_one=False)
    sch.set_timesteps(50)
    out = {}
    for B in images:
        smp = CapturedSampler(unet, sch, B, 64, 64, 77, 7.5)
        g = torch.Generator().manual_seed(7)
        ids_host = torch.randint(0, 49408, (2 * B, 77), generator=g).pin_memory()
        lat_host = torch.randn(B, 4, 64, 64, generator=g).pin_memory()
        img_host = torch.empty(B, 512, 512, 3, dtype=torch.uint8).pin_memory()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

        def once():
            with torch.no_grad():
                ev[0].record()
                ctx2 = clip(ids_host.to(dev, non_blocking=True))[0]
                ev[1].record()
                lat = smp.run(lat_host.to(dev, non_blocking=True), ctx2)
                ev[2].record()
                img = vae.decode(lat / 0.18215).sample
                img = ((img / 2 + 0.5).clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()
                img_host.copy_(img, non_blocking=True)
                ev[3].record()
                torch.cuda.current_stream().synchronize()

        once()
        once()
        t0 = time.perf_counter()
        parts = [0.0, 0.0, 0.0]
        for _ in range(reps):
            once()
            for i in range(3):
                parts[i] += ev[i].elapsed_time(ev[i + 1]) / reps
        wall_ms = (time.perf_counter() - t0) * 1e3 / reps
        out[f"{B}_images"] = {"images_per_s": B / (wall_ms * 1e-3), "ms_per_call": wall_ms, "clip_ms": parts[0], "denoise_50_steps_ms": parts[1],
                              "vae_decode_ms": parts[2]}
        del smp
    out["what"] = ("text ids -> CLIP -> 50 DDIM steps (CFG 7.5) -> VAE decode -> uint8 512x512 on the host, all b200sd kernels; wall "
                   "clock per call incl. H2D / D2H")
    del clip, vae
    return out


def train_text_leg(dev, world, rank, local, steps=5, warmup=3, B=8, unet=None):
    """BASELINE configs[3]: text-encoder fine-tuning (UNet frozen: our forward + data-gradient-only backward down to the context;
    CLIP text model = b200sd.clip.CLIPTextModel, forward and backward on our kernels; flat-gradient allreduce + fused AdamW in
    trainer.TextEncoderTrainer) at batch 8/GPU."""
    import torch
    from b200sd.clip import CLIPTextModel
    from b200sd.schedulers import DDPMScheduler
    from b200sd.trainer import TextEncoderTrainer
    from b200sd.unet import UNet2DConditionModel
    torch.manual_seed(0)
    if unet is None:
        unet = UNet2DConditionModel().to(dev)
    unet = unet.eval().requires_grad_(False)                                      # finetune_sd.py:391-395
    clip = CLIPTextModel().to(dev).train()                                        # SD v1.x text tower, random init (123.1 M)
    sched = DDPMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    tr = TextEncoderTrainer(clip, unet, sched, lr=1e-5, weight_decay=1e-2)
    g = torch.Generator().manual_seed(1000 + rank)
    x0, noise = torch.randn(B, 4, 64, 64, generator=g).to(dev), torch.randn(B, 4, 64, 64, generator=g).to(dev)
    t, ids = torch.randint(0, 1000, (B,), generator=g).to(dev), torch.randint(0, 49408, (B, 77), generator=g).to(dev)
    last = []

    def step():
        last[:] = [tr.train_step(x0, noise, t, ids)]                               # finetune_sd.py:477-494, 569-570

    ms = _timed_steps(step, steps, warmup, world, dev)
    ms_local = ms
    if world > 1:
        tr.allreduce_enabled = False       # same step, every rank on its local gradient
        ms_local = _timed_steps(step, steps, 1, world, dev)
        tr.allreduce_enabled = True
    n_param = sum(p.numel() for p in clip.parameters())
    _, _, tf_sus, _ = _peaks()
    flops_step = 2 * B * FLOPS_PER_SAMPLE_64
    rec = {"workload": "sd15_text_encoder_finetune_512px", "batch_per_gpu": B, "steps": steps, "warmup": warmup, "n_gpus": world,
           "ms_per_step": ms, "samples_per_s": B * world / (ms * 1e-3), "ms_per_step_without_allreduce": ms_local,
           "exposed_comm_ms": ms - ms_local, "allreduce_bytes_on_wire_per_gpu": int(2 * (world - 1) / world * n_param * 4),
           "tflops_per_gpu": flops_step / (ms * 1e-3) / 1e12, "frac_of_sustained_bf16_peak": flops_step / (ms * 1e-3) / 1e12 / tf_sus,
           "last_loss": float(last[0]), "text_encoder": "b200sd.clip.CLIPTextModel (own kernels, forward + backward)",
           "collective": "NCCL all_reduce(SUM) of the flat fp32 gradient buffer of the 123.1 M CLIP parameters (4 chunks) + fused AdamW"}
    del tr, clip
    return rec


def run_train(args):
    _claim_stdout()
    import torch
    import torch.distributed as dist
    from b200sd import ops
    from b200sd.schedulers import DDPMScheduler
    from b200sd.trainer import Trainer
    from b200sd.unet import UNet2DConditionModel

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if rank == 0:
            v, done, t_total, cores = cpu_oracle_train_samples_per_s(1, max(1, min(args.steps, 2)))
            emit(json.dumps({"impl": "reference", "metric": "unet_finetune_samples_per_s", "value": v, "unit": "samples/s",
                              "n_gpus": args.gpus, "steps": done, "warmup": 0, "ms_per_step": 1e3 * t_total / done,
                              "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                              "config": {"workload": "sd15_unet_finetune_512px", "batch_per_gpu": 1},
                              "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                                               "sample": f"{done} optimizer steps at batch 1 (fp32 oracle + torch autograd + AdamW)"},
                              "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                              "gpu_launches": 0}))
        return
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch if args.batch > 1 else 8
    torch.manual_seed(0)                                   # identical initial weights on every rank
    unet = UNet2DConditionModel().to(dev)
    sched = DDPMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    tr = Trainer(unet, sched, lr=1e-5, weight_decay=1e-2, optim_bits=args.optim_bits)
    g = torch.Generator().manual_seed(1000 + rank)
    host = dict(x0=torch.randn(B, 4, 64, 64, generator=g).pin_memory(), noise=torch.randn(B, 4, 64, 64, generator=g).pin_memory(),
                t=torch.randint(0, 1000, (B,), generator=g).pin_memory(), ctx=torch.randn(B, 77, 768, generator=g).pin_memory())
    d = {k: v.to(dev) for k, v in host.items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        tr.train_step(d["x0"], d["noise"], d["t"], d["ctx"])
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ops.launch_count()
    e0.record()
    for _ in range(args.steps):
        loss = tr.train_step(d["x0"], d["noise"], d["t"], d["ctx"])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    launches = ops.launch_count() - l0
    # end to end: host batches in, loss value out, every step
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        dd = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        loss_val = float(tr.train_step(dd["x0"], dd["noise"], dd["t"], dd["ctx"]))
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        tt = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(tt[0]), float(tt[1])
    if rank == 0:
        hbm, tf_burst, tf_sus, which = _peaks()
        samples = B * args.steps * world
        step_ms = ms / args.steps
        flops_step = 3 * B * FLOPS_PER_SAMPLE_64          # SURVEY.md 8(d): fwd + dgrad + wgrad, per GPU
        achieved = flops_step / (step_ms * 1e-3) / 1e12
        n_param = sum(p.numel() for p in unet.parameters())
        line = {"metric": "unet_finetune_samples_per_s", "value": samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "sd15_unet_finetune_512px", "batch_per_gpu": B, "latent": "4x64x64", "context": "77x768",
                           "step": "add_noise + UNet fwd + MSE + bwd (dgrad + wgrad) + bucketed NCCL allreduce + fused AdamW",
                           "optimizer": ("block-wise 8-bit AdamW (bnb.optim.AdamW8bit semantics, the reference's default)"
                                         if args.optim_bits == 8 else "AdamW, fp32 moments (torch.optim.AdamW semantics)"),
                           "weights": "random-init SD v1.5 UNet (859.5M params), fp32 master + bf16 tensor-core copy",
                           "allreduce_bytes_per_gpu": int(2 * (world - 1) / world * n_param * 4), "last_loss": loss_val,
                           "l2": "no flush: 7.4 GB of saved activations + 8.6 GB of parameter state stream through the 126 MB L2 every step"},
                "e2e": {"value": samples / (e2e_ms * 1e-3), "unit": "samples/s",
                        "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host.values())), "d2h_bytes_per_step": 4},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "whole step (forward + backward GEMM / conv / attention)", "achieved": achieved,
                             "peak": tf_sus, "unit": "TFLOP/s", "frac": achieved / tf_sus, "peak_kind": f"bf16 sustained, {which}",
                             "flops_per_step": flops_step, "traffic": None}}
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# text-encoder fine-tuning (BASELINE config 4): UNet frozen (our forward + dgrad-only backward down to the context),
# CLIP text encoder = b200sd.clip.CLIPTextModel (SURVEY.md 8f N3: forward + backward on our kernels), flat-gradient allreduce
# ---------------------------------------------------------------------------------------------------
def run_train_text(args):
    _claim_stdout()
    import torch
    import torch.distributed as dist
    from b200sd import ops
    from b200sd.clip import CLIPTextModel
    from b200sd.schedulers import DDPMScheduler
    from b200sd.trainer import TextEncoderTrainer
    from b200sd.unet import UNet2DConditionModel

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch if args.batch > 1 else 8
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(dev).eval().requires_grad_(False)            # finetune_sd.py:391-395
    clip = CLIPTextModel().to(dev).train()
    sched = DDPMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    g = torch.Generator().manual_seed(1000 + rank)
    host = dict(x0=torch.randn(B, 4, 64, 64, generator=g).pin_memory(), noise=torch.randn(B, 4, 64, 64, generator=g).pin_memory(),
                t=torch.randint(0, 1000, (B,), generator=g).pin_memory(), ids=torch.randint(0, 49408, (B, 77), generator=g).pin_memory())
    d = {k: v.to(dev) for k, v in host.items()}

    tr = TextEncoderTrainer(clip, unet, sched, lr=1e-5, weight_decay=1e-2)

    def step(b):
        return tr.train_step(b["x0"], b["noise"], b["t"], b["ids"])                # finetune_sd.py:477-494, 569-570

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(d)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ops.launch_count()
    e0.record()
    for _ in range(args.steps):
        step(d)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    launches = ops.launch_count() - l0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss_val = float(step({k: v.to(dev, non_blocking=True) for k, v in host.items()}))
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        tt = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(tt[0]), float(tt[1])
    if rank == 0:
        hbm, tf_burst, tf_sus, which = _peaks()
        samples = B * args.steps * world
        step_ms = ms / args.steps
        flops_step = 2 * B * FLOPS_PER_SAMPLE_64          # SURVEY.md 8(d): UNet fwd + dgrad (CLIP ~0.3 % on top)
        achieved = flops_step / (step_ms * 1e-3) / 1e12
        emit(json.dumps({
            "metric": "text_encoder_finetune_samples_per_s", "value": samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "sd15_text_encoder_finetune_512px", "batch_per_gpu": B, "latent": "4x64x64", "tokens": 77,
                       "step": "CLIP fwd + add_noise + frozen UNet fwd + MSE + UNet dgrad-only bwd -> d ctx + CLIP bwd + flat-gradient allreduce + fused AdamW (all b200sd kernels)",
                       "last_loss": loss_val},
            "e2e": {"value": samples / (e2e_ms * 1e-3), "unit": "samples/s",
                    "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host.values())), "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "whole step (UNet forward + data-gradient backward)", "achieved": achieved,
                         "peak": tf_sus, "unit": "TFLOP/s", "frac": achieved / tf_sus, "peak_kind": f"bf16 sustained, {which}",
                         "flops_per_step": flops_step, "traffic": None}}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=1, help="images per GPU (UNet batch = 2x with CFG)")
    ap.add_argument("--lanes", type=int, default=0, help="concurrent launch chains of the captured step (0 = library default)")
    ap.add_argument("--portrait", action="store_true", help="512x768 book-cover geometry (config 5)")
    ap.add_argument("--total-images", type=int, default=0,
                    help="config 5: shard this many images over the GPUs (strong scaling; overrides --batch)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"], help="fp32 = the accuracy path (engine_fp32.py)")
    ap.add_argument("--impl", default="b200sd", choices=["b200sd", "reference", "library"],
                    help="library = the oracle module in bf16 under eager torch on the GPU (yardstick, sampling workload only)")
    ap.add_argument("--sweep-batches", default="1,2,4,8,16,32,64", help="--workload sweep: total image batches to run")
    ap.add_argument("--workload", default="sample", choices=["sample", "train", "train_text", "sweep"],
                    help="sample = 50-step DDIM + CFG denoising (BASELINE configs[1], the headline); train = fine-tuning step (configs[2])")
    ap.add_argument("--optim-bits", type=int, default=32, choices=[32, 8],
                    help="--workload train: 8 = the reference's default block-wise 8-bit AdamW state (finetune_sd.py:300, 407-410)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-legs", action="store_true", help="skip the fine-tuning sub-records (configs 3 / 4) of the default line")
    ap.add_argument("--no-elementwise", action="store_true", help="skip the elementwise GB/s sub-record")
    ap.add_argument("--dump-ops", default=None, help="write the per-launch timing table to this file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="sampling workload: write what the last timed step returned (rank 0) as DIR/latents.npy (the new "
                         "latents) and DIR/noise_pred.npy (the UNet's [uncond | cond] noise prediction), float32")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "sample" or args.impl != "b200sd"):
        ap.error("--dump-outputs covers the sampling workload of the b200sd implementation")
    if args.workload == "sweep":
        if args.gpus > 1 and "RANK" not in os.environ:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
            raise SystemExit(subprocess.call(cmd))
        return run_sweep(args)
    if args.workload in ("train", "train_text"):
        if args.impl != "reference" and args.gpus > 1 and "RANK" not in os.environ:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29532", os.path.abspath(__file__)] + sys.argv[1:]
            raise SystemExit(subprocess.call(cmd))
        run_train_text(args) if args.workload == "train_text" and args.impl != "reference" else run_train(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.impl == "library":
        run_library(args)
    else:
        if args.gpus > 1 and "RANK" not in os.environ:
            # convenience: self-launch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
            raise SystemExit(subprocess.call(cmd))
        run_ours(args)


# NCCL writes its banner ("NCCL version ...") to stdout; the contract is ONE JSON line there, so its log goes to a file
# (not /dev/stderr: fopen(..., "w") would truncate a redirected log).  Set NCCL_DEBUG_FILE yourself to put it elsewhere.
os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/b200sd_nccl.%h.%p.log")

if __name__ == "__main__":
    main()
