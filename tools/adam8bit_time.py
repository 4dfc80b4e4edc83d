"""adamw8bit_step at 64 Mi parameters (22 B / parameter): time per launch and GB/s."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from b200sd import ops
from b200sd.trainer import create_dynamic_map

dev = torch.device("cuda:0")
E = 64 << 20
p, g = torch.randn(E, device=dev), torch.randn(E, device=dev) * 0.01
wb = torch.empty(E, device=dev, dtype=torch.bfloat16)
c1, c2 = torch.zeros(E, device=dev, dtype=torch.uint8), torch.zeros(E, device=dev, dtype=torch.uint8)
a1, a2 = torch.zeros(E // 2048, device=dev), torch.zeros(E // 2048, device=dev)
q1, q2 = create_dynamic_map(True).to(dev), create_dynamic_map(False).to(dev)
fn = lambda: ops.adamw8bit_step(p, g, c1, c2, a1, a2, q1, q2, None, None, None, wb, 1e-5, 0.9, 0.999, 1e-8, 1e-2, 1, grad_scale=1.0,
                                zero_grad=True)
for _ in range(3):
    fn()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10):
    fn()
e1.record()
torch.cuda.synchronize()
us = e0.elapsed_time(e1) * 100.0
print(f"adamw8bit_step: {us:.1f} us per launch, {22 * E / us / 1e3:.1f} GB/s")
