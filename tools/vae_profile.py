"""In-step per-launch times of the VAE decode / encode plans (plan.profile_plan) on random-init SD v1.x weights."""
import sys, torch
sys.path.insert(0, '.')
from b200sd.vae import AutoencoderKL
torch.manual_seed(0)
vae = AutoencoderKL().to('cuda:0').eval()
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1
z = torch.randn(B, 4, 64, 64, device='cuda:0')
img = torch.randn(B, 3, 512, 512, device='cuda:0')
for kind, fn, key in (("decode", lambda: vae.decode(z), ("dec", B, 64, 64, 0)), ("encode", lambda: vae.encode(img), ("enc", B, 512, 512, 0))):
    fn(); fn()
    eng = vae._engines[key]
    acc, per_op, total = eng.profile(3)
    print(f"== {kind} B={B}: instrumented replay {total:.2f} ms, {len(per_op)} launches")
    for k, v in sorted(acc.items(), key=lambda kv: -kv[1][0]):
        print(f"  {k:10s} {v[0]:8.3f} ms  {v[2]:3d} launches  {v[1] / (v[0] * 1e-3) / 1e12 if v[1] else 0:7.1f} TFLOP/s")
    for name, t, fl in sorted(per_op, key=lambda r: -r[1])[:14]:
        print(f"    {t * 1e3:8.1f} us  {fl / (t * 1e-3) / 1e12 if fl else 0:7.1f} TF/s  {name}")
