"""The 9-channel inpainting UNet on the captured sampler, measured on one GPU:

  * per-step time of a captured 50-step DDIM run (CFG 7.5, 64x64 latents, full-size SD v1.x UNet on random weights: the time does
    not depend on them) at 1 and 8 images, the 4-channel text-to-image graph against the 9-channel inpainting graph, with the
    kernels per step of each.  The two alternate in the same process, `--repeats` times each; CUDA events around the step loop;
  * conv_in per launch at Cin = 4 and 9, UNet batch 2 and 16, 64x64, bf16 output (what the bf16 plan runs), as a CUDA graph of
    100 launches replayed `--repeats` times;
  * the input assembly (sampler_inpaint_input) per launch at 1 and 8 images, without a table (DDIM) and with one (LMS), the same way;
  * one StableDiffusionInpaintPipeline call at 1 image, 512x768 portrait, DDIM 50 steps, output_type "pt" (full-size VAE on random
    weights), host clock around a device synchronize, and the same work split into VAE encode + posterior sample, the denoising
    steps, and VAE decode.

Prints the card name and power limit first.  Writes nothing; redirect stdout to keep the report.

    python tools/inpaint_bench.py [--steps 50] [--repeats 5]
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


def _spread(xs, fmt="{:.4f}"):
    f = lambda v: fmt.format(v)
    return f"median {f(statistics.median(xs))}  min {f(min(xs))}  max {f(max(xs))}  (n={len(xs)})"


def _cond(B, h, w):
    mask = torch.zeros(B, 1, h, w, device=DEV)
    mask[:, :, h // 4: h // 2] = 1.0
    return mask, torch.randn(B, 4, h, w, device=DEV)


def step_times(unets, B, steps, repeats):
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(B, 4, 64, 64, generator=g).to(DEV)
    ctx2 = torch.randn(2 * B, 77, 768, generator=g).to(DEV)
    cond = _cond(B, 64, 64)
    smps = {}
    for name, unet in unets.items():
        sch = DDIMScheduler(**_KW)
        sch.set_timesteps(steps)
        smps[name] = CapturedSampler(unet, sch, B, 64, 64, 77, 7.5)
        smps[name].run(lat, ctx2, cond=cond if name == "inpaint9" else None)       # capture + warm up every graph
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
    print(f"\n## per-step time, {B} image(s), DDIM {steps} steps, 64x64 latents, CFG 7.5 (ms per step)")
    for name, xs in times.items():
        print(f"  {name:9s} {_spread(xs)}   kernels/step {smps[name].kernels_per_step}")
    t4, t9 = statistics.median(times["text2img"]), statistics.median(times["inpaint9"])
    print(f"  inpaint9 / text2img: {t9 / t4:.4f} ({(t9 - t4) * 1e3:+.1f} us per step)")
    del smps
    torch.cuda.empty_cache()


def _graph_us(fn, repeats, reps=100):
    """median and range of the per-launch time of `fn` over `repeats` replays of a CUDA graph of `reps` launches"""
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
    xs = []
    for _ in range(repeats):
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        xs.append(e0.elapsed_time(e1) * 1e3 / reps)
    return xs


def conv_in_times(repeats):
    from b200sd import ops
    from b200sd.packing import pack_conv3x3_f32
    print("\n## conv_in per launch, 64x64, 320 output channels, bf16 out (CUDA graph of 100 launches; us)")
    for N in (2, 16):
        for cin in (4, 9):
            x = torch.randn(N, cin, 64, 64, device=DEV)
            w = pack_conv3x3_f32(torch.randn(320, cin, 3, 3, device=DEV) / 6)
            b = torch.randn(320, device=DEV)
            out = torch.empty(N * 64 * 64, 320, dtype=torch.bfloat16, device=DEV)
            xs = _graph_us(lambda: ops.conv_in(x, w, b, out), repeats)
            print(f"  UNet batch {N:2d}  Cin {cin}  {_spread(xs, '{:.2f}')}   {2 * N * 4096 * 320 * 9 * cin / 1e9:.2f} GFLOP")


def assembly_times(repeats):
    from b200sd import ops
    from b200sd.schedulers import LMSDiscreteScheduler
    sch = LMSDiscreteScheduler(**{k: _KW[k] for k in ("beta_start", "beta_end", "beta_schedule")})
    sch.set_timesteps(50)
    table = torch.tensor(sch.sigma_plan()[0], dtype=torch.float32, device=DEV)
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    print("\n## sampler_inpaint_input per launch, 64x64 latents (CUDA graph of 100 launches; us)")
    for B in (1, 8):
        lat = torch.randn(B, 4, 64, 64, device=DEV)
        mask, masked = _cond(B, 64, 64)
        cond = torch.cat([mask, masked], 1)
        x2 = torch.empty(2 * B, 9, 64, 64, device=DEV)
        nbytes = (lat.numel() + cond.numel() + x2.numel()) * 4
        for name, args in (("no table (DDIM)", ()), ("LMS table", (table, cursor))):
            xs = _graph_us(lambda: ops.sampler_inpaint_input(lat, cond, x2, *args), repeats)
            print(f"  {B} image(s)  {name:15s} {_spread(xs, '{:.2f}')}   {nbytes / 1e6:.2f} MB moved")


def end_to_end(unet, steps, repeats):
    from b200sd import StableDiffusionInpaintPipeline
    from b200sd.pipeline import denoise_loop, latent_mask, prepare_mask_and_masked_image
    from b200sd.schedulers import DDIMScheduler
    from b200sd.vae import AutoencoderKL
    torch.manual_seed(0)
    vae = AutoencoderKL().to(DEV).eval()
    H, W = 768, 512
    g = torch.Generator().manual_seed(1)
    image = (torch.rand(1, 3, H, W, generator=g) * 2 - 1).to(DEV)
    mask_image = torch.zeros(1, 1, H, W, device=DEV)
    mask_image[:, :, H // 4: H // 2] = 1.0                 # the title band
    ctx2 = torch.randn(2, 77, 768, generator=g).to(DEV)
    pipe = StableDiffusionInpaintPipeline(vae=vae, unet=unet, scheduler=DDIMScheduler(**_KW))

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    res = {k: [] for k in ("call", "encode", "steps", "decode")}
    for it in range(repeats + 1):                      # the first round captures every graph
        gen = lambda: torch.Generator(DEV).manual_seed(2)
        call, _ = clock(lambda: pipe(prompt_embeds=ctx2, image=image, mask_image=mask_image, height=H, width=W,
                                     num_inference_steps=steps, generator=gen(), output_type="pt"))
        mask, masked_image = prepare_mask_and_masked_image(image, mask_image)
        t_enc, masked = clock(lambda: 0.18215 * vae.encode(masked_image).latent_dist.sample(gen()))
        cond = torch.cat([latent_mask(mask, H // 8, W // 8), masked], 1)
        lat = torch.randn(1, 4, H // 8, W // 8, generator=gen(), device=DEV)
        t_steps, out = clock(lambda: denoise_loop(unet, pipe.scheduler, lat, ctx2, steps, 7.5, cond=cond))
        t_dec, _ = clock(lambda: vae.decode(out / 0.18215).sample)
        if it:
            for k, v in (("call", call), ("encode", t_enc), ("steps", t_steps), ("decode", t_dec)):
                res[k].append(v)
    print(f"\n## one StableDiffusionInpaintPipeline call, 1 image, {W}x{H} (portrait), DDIM {steps} steps, output_type pt; host "
          "clock around a device synchronize (ms)")
    for k, xs in res.items():
        print(f"  {k:7s} {_spread(xs)}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("inpaint_bench.py needs a CUDA device")
    from b200sd.unet import UNet2DConditionModel
    print(_card())
    print(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    torch.manual_seed(0)
    unets = {"text2img": UNet2DConditionModel().to(DEV).eval(), "inpaint9": UNet2DConditionModel(in_channels=9).to(DEV).eval()}
    for B in (1, 8):
        step_times(unets, B, args.steps, args.repeats)
    conv_in_times(args.repeats)
    assembly_times(args.repeats)
    end_to_end(unets["inpaint9"], args.steps, args.repeats)


if __name__ == "__main__":
    main()
