"""Self-attention forward micro-check (timing + error vs torch fp32) for ncu / A-B runs:
python tools/one_attn.py [B] [S] [d] [ramp]   (ramp > 0 makes the scores grow along the keys: exercises the lazy-max redo)"""
import sys, os; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from b200sd import ops
B = int(sys.argv[1]) if len(sys.argv) > 1 else 2
S = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
d = int(sys.argv[3]) if len(sys.argv) > 3 else 40
ramp = float(sys.argv[4]) if len(sys.argv) > 4 else 0.0
H = 8; C = H * d
torch.manual_seed(0)
qkv = torch.randn(B * S, 3 * C, device='cuda')
if ramp > 0:
    qkv[:, C:2 * C] *= (1.0 + ramp * torch.arange(S, device='cuda').repeat(B) / S)[:, None]
qkv = qkv.bfloat16()
out = torch.empty(B * S, C, device='cuda', dtype=torch.bfloat16)
lse = torch.empty(B, H, S, device='cuda')
def run():
    ops.attention_lse(qkv, qkv, qkv, out, lse, B, H, S, S, d, d ** -0.5, ldq=3 * C, ldk=3 * C, ldv=3 * C, ldo=C, k_off=C, v_off=2 * C)
run(); torch.cuda.synchronize()
q, k, v = [t.reshape(B, S, H, d).permute(0, 2, 1, 3).float() for t in qkv.split(C, dim=1)]
sc = (q @ k.transpose(-1, -2)) * d ** -0.5
ref = (torch.softmax(sc, -1) @ v).permute(0, 2, 1, 3).reshape(B * S, C)
ref_lse = torch.logsumexp(sc, -1) * 1.4426950408889634
err = (out.float() - ref).abs().max().item() / ref.abs().max().item()
lerr = (lse - ref_lse).abs().max().item()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
best = 1e9
for i in range(5):
    e0.record()
    for _ in range(4): run()
    e1.record(); torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1) / 4)
fl = 4.0 * B * H * S * S * d
print(f"attention B{B} S{S} d{d} ramp{ramp}: {best * 1e3:.1f} us "
      f"{fl / best / 1e9:.0f} TF/s  max-rel err {err:.2e}  lse err {lerr:.2e}")
