"""Launch-sequence fingerprint of every engine's plan: the exact sequence of C-ABI calls with their arguments, buffer addresses
replaced by the index of the call that first used them.  Two builds whose JSON is identical issue the same kernels with the
same arguments over the same buffer-aliasing pattern, so they compute the same bits.

    python tools/plan_fingerprint.py OUT.json        (needs a GPU: the plans run once, eagerly, on cuda:0)

Random-init SD v1.5 weights (seed 0); only public constructors are used, so the script runs unchanged on older commits."""
import ctypes as C
import json
import sys

import torch

sys.path.insert(0, ".")
from b200sd import ops                                                      # noqa: E402
from b200sd._lib import SIGNATURES, DgradArgs, GemmArgs, WgradArgs          # noqa: E402

_STRUCTS = (GemmArgs, DgradArgs, WgradArgs)


class Recorder:
    """Stands in for ops.lib(): forwards every call to the library and, while `calls` is a list, appends (symbol, args)."""

    def __init__(self, real):
        self.real, self.calls, self.ptrs = real, None, {}

    def _ptr(self, v):
        if not v:
            return None
        return "p%d" % self.ptrs.setdefault(int(v), len(self.calls))

    def _arg(self, t, v):
        if t is C.c_void_p:
            return self._ptr(v)
        if isinstance(v, float):
            return float(C.c_float(v).value) if t is C.c_float else v
        obj = getattr(v, "_obj", None)           # C.byref(struct)
        if isinstance(obj, _STRUCTS):
            return {f: (self._ptr(getattr(obj, f)) if ft is C.c_void_p else getattr(obj, f)) for f, ft in obj._fields_}
        return v if isinstance(v, (int, type(None))) else repr(v)

    def __getattr__(self, name):
        fn = getattr(self.real, name)
        argtypes = SIGNATURES[name][1]

        def call(*args):
            if self.calls is not None:
                self.calls.append([name] + [self._arg(t, v) for t, v in zip(argtypes, args)])
            return fn(*args)
        return call

    def record(self, run):
        self.calls, self.ptrs = [], {}
        try:
            run()
            torch.cuda.synchronize()
            return self.calls
        finally:
            self.calls = None


def counters(eng, names):
    out = {}
    for n in names:
        v = eng
        for part in n.split("."):
            v = getattr(v, part, None)
        if v is not None:
            out[n] = list(v) if isinstance(v, tuple) else v
    return out


def main(path):
    from b200sd.clip import ClipEngine, ClipFlat, CLIPTextModel
    from b200sd.engine import Engine
    from b200sd.engine_fp32 import EngineF32
    from b200sd.train import FlatParams, TrainEngine
    from b200sd.unet import UNet2DConditionModel
    from b200sd.vae import AutoencoderKL, VaeDecodeEngine, VaeEncodeEngine

    rec = Recorder(ops.lib())
    ops.lib = lambda: rec
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    unet = UNet2DConditionModel().to(dev).eval()
    unet._ensure_packed()
    g = torch.Generator(device=dev).manual_seed(0)
    res = {}

    def unet_inputs(N, H, W):
        return (torch.randn(N, 4, H, W, device=dev, generator=g), 500.0,
                torch.randn(N, 77, 768, device=dev, generator=g))

    def infer(key, cls, N, H, W):
        eng = cls(unet, N, H, W, 77, dev)
        x, t, ctx = unet_inputs(N, H, W)
        calls = rec.record(lambda: eng.run(x, t, ctx, use_graph=False))
        eng.run(x, t, ctx, use_graph=True)                 # for kernels_per_graph
        res[key] = dict(calls=calls, counters=counters(eng, ["activation_bytes", "pool.total", "kernels_per_graph"]))
        if cls is Engine:
            res[key]["meta"] = [list(m) for m in eng.plan.meta]

    infer("Engine N2 64x64", Engine, 2, 64, 64)
    infer("Engine N8 64x64", Engine, 8, 64, 64)
    infer("Engine N2 96x64", Engine, 2, 96, 64)
    infer("EngineF32 N2 64x64", EngineF32, 2, 64, 64)

    flat = FlatParams(unet, dev)
    for key, kw in (("TrainEngine N2 64x64 train_weights", dict(train_weights=True)),
                    ("TrainEngine N2 64x64 ctx_grad", dict(train_weights=False, ctx_grad=True))):
        eng = TrainEngine(unet, flat, 2, 64, 64, 77, dev, **kw)
        x, t, ctx = unet_inputs(2, 64, 64)
        d_out = torch.randn(2, 4, 64, 64, device=dev, generator=g)

        def run():
            eng.run_forward(x, t, ctx)
            eng.run_backward(d_out)
        res[key] = dict(calls=rec.record(run), counters=counters(eng, ["saved_bytes", "pool.total"]))
        del eng

    vae = AutoencoderKL().to(dev).eval()
    vae.use_cuda_graph = False
    vae._pack_weights()
    for key, cls, B, H, W, inp in (("VaeDecodeEngine B1 64x64", VaeDecodeEngine, 1, 64, 64, (1, 4, 64, 64)),
                                   ("VaeEncodeEngine B1 512x512", VaeEncodeEngine, 1, 512, 512, (1, 3, 512, 512))):
        eng = cls(vae, B, H, W, dev)
        x = torch.randn(*inp, device=dev, generator=g)
        res[key] = dict(calls=rec.record(lambda: eng.run(x)), counters=counters(eng, ["activation_bytes", "pool.total"]),
                        meta=[list(m) for m in eng.plan.meta])
        del eng

    clip = CLIPTextModel().to(dev)
    cflat = ClipFlat(clip, dev)
    eng = ClipEngine(clip, cflat, 2, 77, dev, train_weights=True)
    eng.use_graph = False
    ids = torch.randint(0, 49407, (2, 77), device=dev, generator=g)
    d_out = torch.randn(2 * 77, 768, device=dev, generator=g)

    def run_clip():
        eng.run_forward(ids)
        eng.run_backward(d_out)
    res["ClipEngine B2 S77 train"] = dict(calls=rec.record(run_clip), counters=counters(eng, ["launches"]))

    with open(path, "w") as f:
        json.dump(res, f, indent=0)
    for k, v in res.items():
        print(f"{k:40s} {len(v['calls']):6d} calls  {v['counters']}")


if __name__ == "__main__":
    main(sys.argv[1])
