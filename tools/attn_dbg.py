import sys, os; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from b200sd import ops
B, S, d = 1, int(sys.argv[1]), int(sys.argv[2]); ramp = float(sys.argv[3])
H = 8; C = H * d
torch.manual_seed(0)
qkv = torch.randn(B * S, 3 * C, device='cuda')
if ramp > 0: qkv[:, C:2 * C] *= (1.0 + ramp * torch.arange(S, device='cuda').repeat(B) / S)[:, None]
qkv = qkv.bfloat16()
out = torch.empty(B * S, C, device='cuda', dtype=torch.bfloat16)
lse = torch.empty(B, H, S, device='cuda')
ops.attention_lse(qkv, qkv, qkv, out, lse, B, H, S, S, d, d ** -0.5, ldq=3 * C, ldk=3 * C, ldv=3 * C, ldo=C, k_off=C, v_off=2 * C)
torch.cuda.synchronize()
q, k, v = [t.reshape(B, S, H, d).permute(0, 2, 1, 3).float() for t in qkv.split(C, dim=1)]
sc = (q @ k.transpose(-1, -2)) * d ** -0.5
ref = (torch.softmax(sc, -1) @ v)            # B H S d
o = out.float().reshape(B, S, H, d).permute(0, 2, 1, 3)
err = (o - ref).abs()
print(f"S{S} d{d} ramp{ramp}: max err {err.max().item():.3e} ref max {ref.abs().max().item():.3f}")
rowerr = err.amax(-1)[0]        # H S
bad = (rowerr > 0.02).nonzero()
print("bad rows:", bad.shape[0], "of", rowerr.numel(), " first:", bad[:8].tolist())
if bad.shape[0]:
    hh, rr = bad[0].tolist()
    print("out", o[0, hh, rr, :8].tolist()); print("ref", ref[0, hh, rr, :8].tolist())
    print("ratio", (o[0, hh, rr, :8] / ref[0, hh, rr, :8]).tolist())
    # which columns are bad
    colerr = err[0, hh, rr]
    print("col err", [round(x, 3) for x in colerr.tolist()])
