"""dgrad / wgrad timing over the training shapes (batch 8, 64x64 latents): tile width / split-K / pair sweeps."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from b200sd import ops
DEV = "cuda:0"
def timeit(fn, reps=10):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(); s = torch.cuda.Stream()
    with torch.cuda.graph(g, stream=s):
        for _ in range(reps): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e9
    for _ in range(3):
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    return best * 1e3
print("== wgrad plain: rows Cout Cin ==")
for (rows, Cout, Cin) in [(32768, 320, 320), (32768, 2560, 320), (32768, 320, 1280), (32768, 960, 320), (8192, 640, 640), (8192, 5120, 640), (2048, 1280, 1280), (2048, 10240, 1280)]:
    dy = torch.randn(rows, Cout, device=DEV).bfloat16(); x = torch.randn(rows, Cin, device=DEV).bfloat16()
    dw = torch.zeros(Cout, Cin, device=DEV)
    row = f"wgrad rows{rows} {Cout}x{Cin}:"
    for bn, sk in ((0, 0), (64, 0), (128, 0), (192, 0), (256, 0), (0, 8), (0, 32)):
        if bn and bn > ((Cin + 63) // 64) * 64: continue
        a = ops.gemm_wgrad(dy, x, dw, block_n=bn, split_k=sk, launch=False)
        t = timeit(lambda: ops.gemm_wgrad_run(a))
        row += f" [bn{bn} sk{sk}] {t:6.1f}us {2 * rows * Cout * Cin / t / 1e6:5.0f}TF"
    print(row, flush=True)
print("== wgrad conv3x3: B H W Cout Cin ==")
for (B, H, W, Cout, Cin) in [(8, 64, 64, 320, 320), (8, 64, 64, 320, 640), (8, 32, 32, 640, 640), (8, 32, 32, 640, 1280), (8, 16, 16, 1280, 1280), (8, 8, 8, 1280, 1280)]:
    rows = B * H * W
    dy = torch.randn(rows, Cout, device=DEV).bfloat16(); x = torch.randn(rows, Cin, device=DEV).bfloat16()
    dw = torch.zeros(Cout, 9 * Cin, device=DEV)
    row = f"wgrad conv {B}x{H}x{W} {Cout}x{Cin}:"
    for bn, sk in ((0, 0), (64, 0), (128, 0), (192, 0), (256, 0), (0, 1), (0, 4)):
        if bn and bn > ((Cin + 63) // 64) * 64: continue
        a = ops.gemm_wgrad(dy, x, dw, conv=(B, H, W), block_n=bn, split_k=sk, launch=False)
        t = timeit(lambda: ops.gemm_wgrad_run(a))
        row += f" [bn{bn} sk{sk}] {t:6.1f}us {2 * rows * Cout * 9 * Cin / t / 1e6:5.0f}TF"
    print(row, flush=True)
print("== dgrad plain: M Cout Cin ==")
for (M, Cout, Cin) in [(32768, 320, 320), (32768, 2560, 320), (32768, 320, 1280), (32768, 960, 320), (8192, 640, 640), (8192, 5120, 640), (2048, 1280, 1280)]:
    dy = torch.randn(M, Cout, device=DEV).bfloat16(); w = torch.randn(Cout, Cin, device=DEV).bfloat16()
    out = torch.empty(M, Cin, device=DEV, dtype=torch.bfloat16)
    row = f"dgrad M{M} {Cout}->{Cin}:"
    for bn, pair in ((0, 0), (64, -1), (128, -1), (192, -1), (256, -1), (128, 1), (256, 1)):
        if bn and bn > ((Cin + 63) // 64) * 64: continue
        a = ops.gemm_dgrad(dy, w, out, block_n=bn, pair=pair, launch=False)
        t = timeit(lambda: ops.gemm_dgrad_run(a))
        row += f" [bn{bn} p{pair}] {t:6.1f}us {2 * M * Cout * Cin / t / 1e6:5.0f}TF"
    print(row, flush=True)
print("== dgrad conv3x3 ==")
for (B, H, W, Cout, Cin) in [(8, 64, 64, 320, 320), (8, 64, 64, 320, 640), (8, 32, 32, 640, 640), (8, 16, 16, 1280, 1280)]:
    M = B * H * W
    dy = torch.randn(M, Cout, device=DEV).bfloat16(); w = torch.randn(Cout, 9 * Cin, device=DEV).bfloat16()
    out = torch.empty(M, Cin, device=DEV, dtype=torch.bfloat16)
    row = f"dgrad conv {B}x{H}x{W} {Cout}->{Cin}:"
    for bn, pair in ((0, 0), (64, -1), (128, -1), (192, -1), (256, -1), (128, 1), (256, 1)):
        if bn and bn > ((Cin + 63) // 64) * 64: continue
        a = ops.gemm_dgrad(dy, w, out, conv=(B, H, W), block_n=bn, pair=pair, launch=False)
        t = timeit(lambda: ops.gemm_dgrad_run(a))
        row += f" [bn{bn} p{pair}] {t:6.1f}us {2 * M * Cout * 9 * Cin / t / 1e6:5.0f}TF"
    print(row, flush=True)
