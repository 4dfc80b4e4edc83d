"""Image-to-image and legacy inpainting on the captured sampler, measured on one GPU:

  * per-step time of a captured run in three modes -- text-to-image (all 50 DDIM steps), img2img and inpaint (strength 0.75:
    the last 37 of the 50 steps) -- at 1 and 8 images (64x64 latents, CFG 7.5, full-size SD v1.x UNet on random weights: the
    time does not depend on them).  The modes alternate in the same process, `--repeats` times each; CUDA events around the
    step loop;
  * `inpaint_blend` alone at the latents' size (CUDA graph of 100 launches): it reads x, x0, z and the mask and writes x,
    5*E*4 bytes, 0.33 MB at 1 image;
  * one `StableDiffusionImg2ImgPipeline` and one `StableDiffusionInpaintPipelineLegacy` call end to end at 1 image, 512x512,
    output_type "pt" (full-size VAE on random weights), host clock around a device synchronize, and the same work split into
    VAE encode + posterior sample, the denoising steps, and VAE decode.

Prints the card name and power limit first.  Writes nothing; redirect stdout to keep the report.

    python tools/img2img_bench.py [--steps 50] [--strength 0.75] [--repeats 5]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

DEV = torch.device("cuda:0")
_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, set_alpha_to_one=False)


def _card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip()


def _spread(xs):
    return f"median {statistics.median(xs):.4f}  min {min(xs):.4f}  max {max(xs):.4f}  (n={len(xs)})"


def step_times(unet, B, steps, strength, repeats):
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(B, 4, 64, 64, generator=g).to(DEV)
    ctx2 = torch.randn(2 * B, 77, 768, generator=g).to(DEV)
    mask = torch.zeros(1, 4, 64, 64, device=DEV)
    mask[:, :, :32] = 1.0
    blend = (lat, torch.randn_like(lat), mask)
    smps = {}
    for name, inpaint in (("text2img", False), ("img2img", False), ("inpaint", True)):
        sch = DDIMScheduler(**_KW)
        start = 0 if name == "text2img" else sch.img2img_start(steps, strength)[0]
        sch.set_timesteps(steps)
        smps[name] = CapturedSampler(unet, sch, B, 64, 64, 77, 7.5, start=start, inpaint=inpaint)
        smps[name].run(lat, ctx2, blend=blend if inpaint else None)         # capture + warm up every graph
    times = {k: [] for k in smps}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(repeats):
            for name, smp in smps.items():
                smp.set_context(ctx2)
                smp.set_latents(lat)
                smp.reset(0)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(smp.n_steps):
                    smp.step()
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / smp.n_steps)
    print(f"\n## per-step time, {B} image(s), DDIM {steps} steps, strength {strength}, 64x64 latents, CFG 7.5 (ms per step)")
    for name, xs in times.items():
        print(f"  {name:9s} {_spread(xs)}   steps {smps[name].n_steps}   kernels/step {smps[name].kernels_per_step}")
    del smps
    torch.cuda.empty_cache()


def blend_time(B, reps=100):
    from b200sd import ops
    from b200sd.schedulers import DDIMScheduler
    sa, sb = DDIMScheduler(**_KW)._noise_tables(DEV)
    x, x0, z, m = (torch.randn(B, 4, 64, 64, device=DEV) for _ in range(4))
    t_table = torch.full((1,), 500.0, device=DEV)
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    fn = lambda: ops.inpaint_blend_table(x, x0, z, m, t_table, cursor, sa, sb)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for _ in range(reps):
            fn()
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = 5 * x.numel() * 4
    print(f"## inpaint_blend_table, {B} image(s): {us:.2f} us per launch, {nbytes / 1e6:.2f} MB "
          f"({nbytes / us / 1e3:.0f} GB/s; the working set sits in L2)")


def end_to_end(unet, steps, strength, repeats):
    from b200sd import StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy
    from b200sd.pipeline import denoise_loop
    from b200sd.schedulers import DDIMScheduler
    from b200sd.vae import AutoencoderKL
    torch.manual_seed(0)
    vae = AutoencoderKL().to(DEV).eval()
    g = torch.Generator().manual_seed(1)
    image = (torch.rand(1, 3, 512, 512, generator=g) * 2 - 1).to(DEV)
    ctx2 = torch.randn(2, 77, 768, generator=g).to(DEV)
    mask = torch.zeros(1, 4, 64, 64, device=DEV)
    mask[:, :, :32] = 1.0
    pipes = {"img2img": (StableDiffusionImg2ImgPipeline(vae=vae, unet=unet, scheduler=DDIMScheduler(**_KW)), {}),
             "inpaint": (StableDiffusionInpaintPipelineLegacy(vae=vae, unet=unet, scheduler=DDIMScheduler(**_KW)),
                         dict(mask_image=mask))}

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    res = {name: {k: [] for k in ("call", "encode", "steps", "decode")} for name in pipes}
    for it in range(repeats + 1):                      # the first round captures every graph
        for name, (pipe, kw) in pipes.items():
            gen = lambda: torch.Generator(DEV).manual_seed(2)
            call, _ = clock(lambda: pipe(prompt_embeds=ctx2, init_image=image, strength=strength, num_inference_steps=steps,
                                         generator=gen(), output_type="pt", **kw))
            sch = pipe.scheduler
            t_enc, init = clock(lambda: 0.18215 * vae.encode(image).latent_dist.sample(gen()))
            t_start, t_noise = sch.img2img_start(steps, strength)
            noise = torch.randn(init.shape, generator=gen(), device=DEV)
            lat = sch.add_noise(init, noise, torch.tensor([t_noise]))
            blend = (init, noise, mask) if kw else None
            t_steps, out = clock(lambda: denoise_loop(unet, sch, lat, ctx2, steps, 7.5, start=t_start, blend=blend))
            t_dec, _ = clock(lambda: vae.decode(out / 0.18215).sample)
            if it:
                for k, v in (("call", call), ("encode", t_enc), ("steps", t_steps), ("decode", t_dec)):
                    res[name][k].append(v)
    print(f"\n## one pipeline call, 1 image, 512x512, DDIM {steps} steps, strength {strength} "
          f"({steps - sch.img2img_start(steps, strength)[0]} executed), output_type pt; host clock around a device synchronize (ms)")
    for name, parts in res.items():
        for k, xs in parts.items():
            print(f"  {name:8s} {k:7s} {_spread(xs)}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--strength", type=float, default=0.75)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("img2img_bench.py needs a CUDA device")
    from b200sd.unet import UNet2DConditionModel
    print(_card())
    print(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(DEV).eval()
    for B in (1, 8):
        step_times(unet, B, args.steps, args.strength, args.repeats)
    print()
    for B in (1, 8):
        blend_time(B)
    end_to_end(unet, args.steps, args.strength, args.repeats)


if __name__ == "__main__":
    main()
