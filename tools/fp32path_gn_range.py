"""How far from zero are the group means of the GroupNorm inputs of the fp32-accuracy path?

The GroupNorm statistics kernels accumulate sums of x and x^2 in fp32 and take var = E[x^2] - E[x]^2, so their error grows with
r = |group mean| / group std (~u r^2 relative in the variance).  This wraps ops.groupnorm_silu_split while EngineF32 runs eager
forwards of the random-init oracle weights (oracle.unet_ref.make_oracle_unet, seed 0) at 64x64 and 96x64 latents, batch 2,
t in {999, 500, 37, 1}, and prints, per call site, the largest r over images, groups and timesteps.

    python tools/fp32path_gn_range.py            (needs a CUDA device)
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    from b200sd import ops
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet

    dev = torch.device("cuda:0")
    oracle = make_oracle_unet(seed=0)
    unet = UNet2DConditionModel()
    unet.load_state_dict(oracle.state_dict(), strict=True)
    unet = unet.to(dev).eval().set_precision("fp32")
    unet.use_cuda_graph = False
    real = ops.groupnorm_silu_split
    sites = {}          # (geometry, call index) -> [signature, max r]
    state = {"geo": None, "i": 0}

    def spy(x0, x1, gamma, beta, out, out_lo, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None, raw_lo=None):
        x = torch.cat([x0, x1], 1) if x1 is not None else x0
        grp = x.double().reshape(batch, hw, groups, -1).permute(0, 2, 1, 3).reshape(batch, groups, -1)
        r = float((grp.mean(-1).abs() / grp.std(-1, unbiased=False)).max())
        key = (state["geo"], state["i"])
        sig = f"hw={hw:5d} C={x0.shape[1]:4d}+{x1.shape[1] if x1 is not None else 0:<4d} silu={int(bool(silu))} eps={eps:g}"
        prev = sites.get(key, [sig, 0.0])
        sites[key] = [sig, max(prev[1], r)]
        state["i"] += 1
        return real(x0, x1, gamma, beta, out, out_lo, batch, hw, groups, eps, silu, raw_out=raw_out, raw_lo=raw_lo)

    ops.groupnorm_silu_split = spy
    try:
        with torch.no_grad():
            for H, W in ((64, 64), (96, 64)):
                g = torch.Generator().manual_seed(H)
                x = torch.randn(2, 4, H, W, generator=g).to(dev)
                ctx = torch.randn(2, 77, 768, generator=g).to(dev)
                for t in (999, 500, 37, 1):
                    state["geo"], state["i"] = f"{H}x{W}", 0
                    unet(x, t, ctx)
    finally:
        ops.groupnorm_silu_split = real
    print(f"GroupNorm inputs of the fp32 path: largest |group mean| / group std per call site "
          f"({torch.cuda.get_device_name(dev)}; random-init oracle weights, seed 0; batch 2; t in 999, 500, 37, 1)")
    worst = 0.0
    for (geo, i), (sig, r) in sorted(sites.items()):
        print(f"{geo:6s} #{i:2d}  {sig}  max r = {r:.3f}")
        worst = max(worst, r)
    print(f"overall max r = {worst:.3f}; envelope max(30, 4 x max) = {max(30.0, 4 * worst):.3g}")


if __name__ == "__main__":
    main()
