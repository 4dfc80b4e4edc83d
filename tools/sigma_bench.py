"""The sigma-space schedulers (LMS, Euler, Euler-ancestral) on the captured sampler, measured on one GPU:

  * per-step time of a captured 50-step run for DDIM (eta = 0) and each of the three schedulers at 1 and 8 images (64x64
    latents, CFG 7.5, full-size SD v1.x UNet on random weights: the time does not depend on them).  The schedulers alternate
    in the same process, `--repeats` times each; CUDA events around the step loop.  kernels/step counts this library's
    launches (the two torch latents copies of the DDIM step are not counted; the sigma step replaces them with one
    sampler_scale_input launch);
  * `cfg_sigma_step_table` (an LMS row of order 4: eps_u, eps_c, x, three history rows read, x and the derivative written,
    8*E*4 bytes) and `sampler_scale_input` (x read, two copies written, 3*E*4 bytes) alone at the latents' size, each in a CUDA
    graph of 100 launches;
  * one StableDiffusionPipeline call end to end at 1 image, 512x512, output_type "pt" (full-size VAE on random weights), host
    clock around a device synchronize: Euler-ancestral at 25 steps next to DDIM at 50.

Prints the card name and power limit first.  Writes nothing; redirect stdout to keep the report.

    python tools/sigma_bench.py [--steps 50] [--repeats 5]
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
_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
_DDIM_KW = dict(_KW, clip_sample=False, set_alpha_to_one=False)


def _card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip()


def _spread(xs):
    return f"median {statistics.median(xs):.4f}  min {min(xs):.4f}  max {max(xs):.4f}  (n={len(xs)})"


def _schedulers():
    from b200sd import schedulers as S
    return {"ddim": lambda: S.DDIMScheduler(**_DDIM_KW), "lms": lambda: S.LMSDiscreteScheduler(**_KW),
            "euler": lambda: S.EulerDiscreteScheduler(**_KW), "euler_a": lambda: S.EulerAncestralDiscreteScheduler(**_KW)}


def step_times(unet, B, steps, repeats):
    from b200sd.sampler import CapturedSampler
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(B, 4, 64, 64, generator=g).to(DEV)
    ctx2 = torch.randn(2 * B, 77, 768, generator=g).to(DEV)
    smps = {}
    for name, make in _schedulers().items():
        sch = make()
        sch.set_timesteps(steps)
        smps[name] = CapturedSampler(unet, sch, B, 64, 64, 77, 7.5)
        smps[name].run(lat, ctx2, generator=torch.Generator(DEV).manual_seed(0))      # capture + warm up every graph
    times = {k: [] for k in smps}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(repeats):
            for name, smp in smps.items():
                smp.set_context(ctx2)
                smp.set_latents(lat * smp.scheduler.init_noise_sigma)
                smp.draw_noise(torch.Generator(DEV).manual_seed(0))
                smp.reset(0)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(smp.n_steps):
                    smp.step()
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / smp.n_steps)
    print(f"\n## per-step time, {B} image(s), {steps} steps, 64x64 latents, CFG 7.5 (ms per step)")
    for name, xs in times.items():
        print(f"  {name:8s} {_spread(xs)}   kernels/step {smps[name].kernels_per_step}")
    del smps
    torch.cuda.empty_cache()


def _graph_time(fn, reps=100):
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
    return e0.elapsed_time(e1) * 1e3 / reps


def kernel_times(B):
    from b200sd import ops
    from b200sd.schedulers import LMSDiscreteScheduler
    sch = LMSDiscreteScheduler(**_KW)
    sch.set_timesteps(50)
    rows, _ = sch.sigma_plan()
    table = torch.tensor(rows, dtype=torch.float32, device=DEV)
    assert all(s >= 0 for s in rows[10][5:9])                     # order 4: three history rows and the derivative slot
    shape = (B, 4, 64, 64)
    E = B * 4 * 64 * 64
    eu, ec, x = (torch.randn(shape, device=DEV) for _ in range(3))
    ring = torch.randn(4, E, device=DEV)
    x2 = torch.empty((2 * B, 4, 64, 64), device=DEV)
    cursor = torch.tensor([0, 10], dtype=torch.int32, device=DEV)
    # the same row every launch: x drifts by O(1) per launch and stays finite over the 100 launches
    us_step = _graph_time(lambda: ops.cfg_sigma_step_table(eu, ec, x, ring, None, 7.5, table, cursor))
    us_scale = _graph_time(lambda: ops.sampler_scale_input(x, x2, table, cursor))
    for name, us, nbytes in (("cfg_sigma_step_table (LMS, order 4)", us_step, 8 * E * 4),
                             ("sampler_scale_input", us_scale, 3 * E * 4)):
        print(f"## {name}, {B} image(s): {us:.2f} us per launch, {nbytes / 1e6:.2f} MB "
              f"({nbytes / us / 1e3:.0f} GB/s; the working set sits in L2)")


def end_to_end(unet, repeats):
    from b200sd import StableDiffusionPipeline
    from b200sd.vae import AutoencoderKL
    torch.manual_seed(0)
    vae = AutoencoderKL().to(DEV).eval()
    ctx2 = torch.randn(2, 77, 768, generator=torch.Generator().manual_seed(1)).to(DEV)
    S = _schedulers()
    runs = {"ddim_50": (StableDiffusionPipeline(vae=vae, unet=unet, scheduler=S["ddim"]()), 50),
            "euler_a_25": (StableDiffusionPipeline(vae=vae, unet=unet, scheduler=S["euler_a"]()), 25)}

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    res = {k: [] for k in runs}
    for it in range(repeats + 1):                      # the first round captures every graph
        for name, (pipe, n) in runs.items():
            ms = clock(lambda: pipe(prompt_embeds=ctx2, num_inference_steps=n, generator=torch.Generator(DEV).manual_seed(2),
                                    output_type="pt"))
            if it:
                res[name].append(ms)
    print("\n## one StableDiffusionPipeline call, 1 image, 512x512, output_type pt; host clock around a device synchronize (ms)")
    for name, xs in res.items():
        print(f"  {name:10s} {_spread(xs)}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sigma_bench.py needs a CUDA device")
    from b200sd.unet import UNet2DConditionModel
    print(_card())
    print(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(DEV).eval()
    for B in (1, 8):
        step_times(unet, B, args.steps, args.repeats)
    print()
    for B in (1, 8):
        kernel_times(B)
    end_to_end(unet, args.repeats)


if __name__ == "__main__":
    main()
