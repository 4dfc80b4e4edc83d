"""Eager vs CUDA-graph replay consistency of one UNet forward (detects launch-ordering races)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from b200sd.unet import UNet2DConditionModel
dev = "cuda:0"
torch.manual_seed(0)
m = UNet2DConditionModel().to(dev).eval()
g = torch.Generator().manual_seed(1)
x = torch.randn(2, 4, 64, 64, generator=g).to(dev); ctx = torch.randn(2, 77, 768, generator=g).to(dev)
t = torch.tensor([980, 20], device=dev)
with torch.no_grad():
    m.use_cuda_graph = False
    e1 = m(x, t, ctx).sample; e2 = m(x, t, ctx).sample
    m.use_cuda_graph = True
    g1 = m(x, t, ctx).sample; g2 = m(x, t, ctx).sample; g3 = m(x, t, ctx).sample
s = float(e1.abs().max())
print("scale", s)
for n, a, b in (("eager-eager", e1, e2), ("eager-graph", e1, g1), ("graph-graph", g1, g2), ("graph-graph2", g2, g3)):
    print(f"{n:14s} max abs diff {float((a - b).abs().max()):.3e}  rel {float((a - b).abs().max()) / s:.3e}")
