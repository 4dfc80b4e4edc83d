"""Ancestral sampling on the captured sampler (DDPMScheduler; DDIMScheduler with eta > 0), measured on one GPU:

  * per-step time of a 50-step captured run in three modes -- DDIM eta = 0, DDIM eta = 1, DDPM -- at 1 and 8 images
    (64x64 latents, CFG 7.5, full-size SD v1.x UNet on random weights: the time does not depend on them).  The modes alternate
    in the same process, `--repeats` times each; CUDA events around the step loop;
  * the host-side fill of the noise table (`CapturedSampler.draw_noise`) per run, with a CPU and with a CUDA generator;
  * `cfg_ancestral_step` at 64 Mi fp32 elements (every operand larger than the L2): algorithmic bytes 5*E*4 (read eps_u,
    eps_c, x, z; write x'), next to `cfg_ddim_step` (4*E*4) and a device-to-device copy (2*E*4).

Prints the card name and power limit first.  Writes nothing; redirect stdout to keep the report.

    python tools/ancestral_bench.py [--steps 50] [--repeats 5]
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


def _card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip()


def _spread(xs):
    return f"median {statistics.median(xs):.4f}  min {min(xs):.4f}  max {max(xs):.4f}  (n={len(xs)})"


def _samplers(unet, B, steps):
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler, DDPMScheduler
    out = {}
    for name, sch, eta in (("ddim_eta0", DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=False), 0.0),
                           ("ddim_eta1", DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=False), 1.0),
                           ("ddpm", DDPMScheduler(num_train_timesteps=1000, **_KW), 0.0)):
        sch.set_timesteps(steps)
        out[name] = CapturedSampler(unet, sch, B, 64, 64, 77, 7.5, eta=eta)
    return out


def step_times(unet, B, steps, repeats):
    smps = _samplers(unet, B, steps)
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(B, 4, 64, 64, generator=g).to(DEV)
    ctx2 = torch.randn(2 * B, 77, 768, generator=g).to(DEV)
    for smp in smps.values():              # capture + warm up every graph
        smp.run(lat, ctx2, generator=torch.Generator(DEV).manual_seed(0))
    times = {k: [] for k in smps}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(repeats):
            for name, smp in smps.items():
                smp.set_context(ctx2)
                smp.set_latents(lat)
                if smp.noise.shape[0]:
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
        print(f"  {name:10s} {_spread(xs)}   kernels/step {smps[name].kernels_per_step}")
    noise_fill = {}
    smp = smps["ddpm"]
    for label, mk in (("cpu_generator", lambda: torch.Generator().manual_seed(0)),
                      ("cuda_generator", lambda: torch.Generator(DEV).manual_seed(0))):
        xs = []
        for _ in range(repeats + 1):
            gen = mk()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            smp.draw_noise(gen)
            torch.cuda.synchronize()
            xs.append((time.perf_counter() - t0) * 1e3)
        noise_fill[label] = xs[1:]          # the first fill pays one-time set-up
    print(f"## draw_noise per run, DDPM {smp.noise.shape[0]} noise rows x {smp.noise.shape[1]} floats "
          f"({smp.noise.numel() * 4 / 1e6:.2f} MB), host clock around a device synchronize (ms)")
    for label, xs in noise_fill.items():
        print(f"  {label:15s} {_spread(xs)}")
    del smps
    torch.cuda.empty_cache()


def bandwidth(repeats):
    from b200sd import ops
    E = 64 << 20
    mk = lambda: torch.randn(E, device=DEV)
    eu, ec, x, z, o = (mk() for _ in range(5))

    def timed(fn, reps=10):
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

    cases = {
        "copy": (lambda: o.copy_(x), 2 * E * 4, "read x; write out"),
        "cfg_ddim_step": (lambda: ops.cfg_ddim_step(eu, ec, x, 7.5, 0.9, 0.43, 0.92, 0.39, out=o), 4 * E * 4,
                          "read eps_u, eps_c, x; write x'"),
        "cfg_ancestral_step": (lambda: ops.cfg_ancestral_step(eu, ec, x, z, 7.5, 0.9, 0.43, 0.7, 0.2, 0.1, 0.05, True, out=o),
                               5 * E * 4, "read eps_u, eps_c, x, z; write x'"),
    }
    res = {k: [] for k in cases}
    for _ in range(repeats):
        for k, (fn, _, _) in cases.items():
            res[k].append(timed(fn))
    copy_gbs = cases["copy"][1] / statistics.median(res["copy"]) / 1e9
    print(f"\n## elementwise bandwidth at E = 64 Mi fp32 elements (CUDA graph of 10 launches, {repeats} repeats, median)")
    for k, (_, nbytes, what) in cases.items():
        t = statistics.median(res[k])
        gbs = nbytes / t / 1e9
        print(f"  {k:20s} {t * 1e6:9.1f} us  {gbs:7.0f} GB/s  {gbs / copy_gbs:5.2f} x copy   bytes {nbytes / 2**20:.0f} MiB ({what})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ancestral_bench.py needs a CUDA device")
    from b200sd.unet import UNet2DConditionModel
    print(_card())
    print(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(DEV).eval()
    for B in (1, 8):
        step_times(unet, B, args.steps, args.repeats)
    bandwidth(args.repeats)


if __name__ == "__main__":
    main()
