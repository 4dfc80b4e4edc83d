"""Per-kernel-kind device time of one training step (forward + backward plans of train.TrainEngine), CUDA-event
timed per plan entry on the launching stream.  Usage: python tools/profile_train.py [batch] [latent_h] [latent_w]"""
import collections
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from b200sd import ops
from b200sd.unet import UNet2DConditionModel


def kind_of(fn):
    names = fn.__code__.co_names
    for n in ("gemm_dgrad_run", "gemm_wgrad_run", "gemm_run"):
        if n in names:
            return n
    for n in names:
        if hasattr(ops, n) and n not in ("check", "lib", "C"):
            return n
    return "torch:" + "/".join(names[:2])


def main():
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    h = int(sys.argv[2]) if len(sys.argv) > 2 else 64
    w = int(sys.argv[3]) if len(sys.argv) > 3 else 64
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(dev).train()
    unet.enable_direct_gradients()
    x = torch.randn(N, 4, h, w, device=dev)
    noise = torch.randn_like(x)
    ctx = torch.randn(N, 77, 768, device=dev)
    t = torch.randint(0, 1000, (N,), device=dev)
    for _ in range(2):
        ops.mse_loss(unet(x, t, ctx).sample, noise).backward()
    torch.cuda.synchronize()
    eng = next(iter(unet._train_engines.values()))
    print(f"saved activations {eng.saved_bytes / 2**30:.2f} GiB, backward scratch {eng.pool.total / 2**30:.2f} GiB, "
          f"fwd entries {len(eng.fwd)}, bwd entries {len(eng.bwd)}")
    # whole-step timing
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    reps = 3
    tf = tb = 0.0
    for _ in range(reps):
        e0.record()
        out = unet(x, t, ctx).sample
        loss = ops.mse_loss(out, noise)
        e1.record()
        loss.backward()
        e2.record()
        torch.cuda.synchronize()
        tf += e0.elapsed_time(e1) / reps
        tb += e1.elapsed_time(e2) / reps
    flops = 0.8033e12 * N * (h * w) / 4096
    print(f"batch {N} {h}x{w}: forward {tf:.2f} ms, backward {tb:.2f} ms, total {tf + tb:.2f} ms -> "
          f"{3 * flops / (tf + tb) / 1e9:.1f} TFLOP/s (3x fwd FLOPs)")
    for label, plan in (("forward", eng.fwd), ("backward", eng.bwd)):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(plan) + 1)]
        if label == "backward":
            eng.d_tproj.zero_()
        evs[0].record()
        for i, op in enumerate(plan):
            op()
            evs[i + 1].record()
        torch.cuda.synchronize()
        acc = collections.defaultdict(lambda: [0.0, 0])
        for i, op in enumerate(plan):
            k = kind_of(op)
            acc[k][0] += evs[i].elapsed_time(evs[i + 1])
            acc[k][1] += 1
        tot = sum(v[0] for v in acc.values())
        print(f"--- {label}: {tot:.2f} ms (eager launches, includes host gaps)")
        for k, (ms, n) in sorted(acc.items(), key=lambda kv: -kv[1][0]):
            print(f"  {k:28s} {ms:8.3f} ms  {n:5d} launches  {100 * ms / tot:5.1f} %")


if __name__ == "__main__":
    main()
