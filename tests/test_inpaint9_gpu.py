"""The 9-channel inpainting UNet and StableDiffusionInpaintPipeline on the GPU: conv_in at Cin = 9 against float64, the captured
step's input assembly against cat + scale_model_input bit for bit, the exact wiring check (a 9-channel UNet with zero weights on
the extra channels is the 4-channel UNet, forward and captured run), the full-size UNet on both plans and the captured
sampler against the fp32 oracle (oracle/inpaint_ref.py) and the per-call loop, every scheduler on the reduced-width net, the
pipeline end to end, and the kernels per captured step."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
RHO = 2.0 ** -8
BAND = 128

from oracle import ancestral_ref as A
from oracle import inpaint_ref as P9
from oracle import schedulers_ref as R
from oracle import sigma_ref as S

_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
_DDIM_KW = dict(_KW, clip_sample=False, set_alpha_to_one=False)
KINDS = ("ddim", "plms", "ddpm", "ddim_eta1", "lms", "euler", "euler_ancestral")


def _cos(a, b):
    return float(F.cosine_similarity(a.float().cpu().flatten(), b.float().cpu().flatten(), dim=0))


def _sched(kind):
    """(ours, oracle, eta), set_timesteps not yet called"""
    from b200sd import schedulers as B
    if kind == "plms":
        return B.PNDMScheduler(**_KW, skip_prk_steps=True), R.PNDMSchedulerRef(skip_prk_steps=True), 0.0
    if kind == "ddpm":
        return B.DDPMScheduler(num_train_timesteps=1000, **_KW), A.DDPMSchedulerRef(), 0.0
    if kind in ("ddim", "ddim_eta1"):
        return B.DDIMScheduler(**_DDIM_KW), A.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), float(kind == "ddim_eta1")
    ours, ref = {"lms": (B.LMSDiscreteScheduler, S.LMSDiscreteSchedulerRef),
                 "euler": (B.EulerDiscreteScheduler, S.EulerDiscreteSchedulerRef),
                 "euler_ancestral": (B.EulerAncestralDiscreteScheduler, S.EulerAncestralDiscreteSchedulerRef)}[kind]
    return ours(**_KW), ref(**_KW), 0.0


def _nan(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


# ---------------------------------------------------------------------------------------------------
# the kernels
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("odt", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("H,W", [(64, 64), (96, 64), (5, 7)])
@pytest.mark.parametrize("B", [1, 2, 8, 16])
def test_conv_in_nine_channels_vs_float64(B, H, W, odt):
    from b200sd import ops
    from b200sd.packing import pack_conv3x3_f32
    Cin, Cout = 9, 320
    g = torch.Generator(device=DEV).manual_seed(B * 100 + H)
    x = torch.randn(B, Cin, H, W, generator=g, device=DEV)
    w = torch.randn(Cout, Cin, 3, 3, generator=g, device=DEV) / 9
    b = torch.randn(Cout, generator=g, device=DEV)
    n = B * H * W
    out = _nan((n + BAND, Cout), odt)
    ops.conv_in(x, pack_conv3x3_f32(w), b, out[:n])
    torch.cuda.synchronize()
    assert torch.isnan(out[n:]).all(), "conv_in wrote past its output"
    got = out[:n].reshape(B, H, W, Cout).double()
    ref = F.conv2d(x.double(), w.double(), b.double(), padding=1).permute(0, 2, 3, 1)
    mag = (F.conv2d(x.double().abs(), w.double().abs(), padding=1) + b.double().abs()[:, None, None]).permute(0, 2, 3, 1)
    rho = RHO if odt == torch.bfloat16 else 0.0
    r = float(((got - ref).abs() / (rho * ref.abs() + 40 * U * mag)).max())
    print(f"conv_in Cin=9 B={B} {H}x{W} -> {odt}: worst {r:.3f} of the 40 u bar")
    assert r <= 1.0


@pytest.mark.parametrize("hw", [(64, 48), (5, 7)])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("kind", ["ddim", "lms", "euler_ancestral"])
def test_input_assembly_equals_cat_then_scale_bit_for_bit(kind, B, hw):
    """No table (DDIM, PLMS, DDPM: a copy), and every row of an LMS and an Euler-a table (a true division)"""
    from b200sd import ops
    h, w = hw
    ours = _sched(kind)[0]
    ours.set_timesteps(50)
    g = torch.Generator(device=DEV).manual_seed(B + h)
    lat = torch.randn(B, 4, h, w, generator=g, device=DEV) * 14
    mask = (torch.rand(B, 1, h, w, generator=g, device=DEV) > 0.5).float()
    cond = torch.cat([mask, torch.randn(B, 4, h, w, generator=g, device=DEV)], 1)
    x2 = _nan((2 * B, 9, h, w), torch.float32)
    if kind == "ddim":
        ops.sampler_inpaint_input(lat, cond, x2)
        assert torch.equal(x2, torch.cat([torch.cat([lat] * 2), torch.cat([cond] * 2)], 1))
        return
    table = torch.tensor(ours.sigma_plan()[0], dtype=torch.float32, device=DEV)
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    for k, t in enumerate(ours.timesteps.tolist()):
        cursor[1] = k
        ops.sampler_inpaint_input(lat, cond, x2, table, cursor)
        want = ours.scale_model_input(torch.cat([torch.cat([lat] * 2), torch.cat([cond] * 2)], 1), t)
        assert torch.equal(x2, want), f"row {k}"


# ---------------------------------------------------------------------------------------------------
# the full-size network
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def full():
    """(fp32 oracle 9-channel UNet on the CPU, ours on the GPU)"""
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    oracle = make_oracle_unet(seed=0, in_channels=9)
    ours = UNet2DConditionModel(in_channels=9)
    ours.load_state_dict(oracle.state_dict(), strict=True)
    return oracle, ours.to(DEV).eval()


def _cond(B, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    mask = torch.zeros(B, 1, h, w)
    mask[:, :, h // 4: h // 2] = 1.0                    # repaint a band, as for a title
    return torch.cat([mask, 0.8 * torch.randn(B, 4, h, w, generator=g)], 1)


def test_zero_extra_channels_reproduce_the_four_channel_unet_bit_for_bit(full):
    """conv_in accumulates bias first, then tap-major channel-minor: zero weights on channels 4..8 add exact zeros, so the
    forward and a captured 50-step DDIM run of the 9-channel UNet equal the 4-channel UNet's"""
    from b200sd.pipeline import denoise_loop
    from b200sd.unet import UNet2DConditionModel
    _, nine = full
    four = UNet2DConditionModel()
    sd = {k: v.detach().cpu() for k, v in nine.state_dict().items()}
    sd["conv_in.weight"] = sd["conv_in.weight"][:, :4].clone()
    four.load_state_dict(sd, strict=True)
    four = four.to(DEV).eval()
    zeroed = UNet2DConditionModel(in_channels=9)
    sd9 = {k: v.detach().cpu() for k, v in nine.state_dict().items()}
    sd9["conv_in.weight"] = sd9["conv_in.weight"].clone()
    sd9["conv_in.weight"][:, 4:] = 0.0
    zeroed.load_state_dict(sd9, strict=True)
    zeroed = zeroed.to(DEV).eval()
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(2, 4, 64, 64, generator=g)
    ctx = torch.randn(2, 77, 768, generator=g)
    cond = _cond(2, 64, 64, 4)
    with torch.no_grad():
        want = four(lat.to(DEV), 500, ctx.to(DEV)).sample
        got = zeroed(torch.cat([lat, cond], 1).to(DEV), 500, ctx.to(DEV)).sample
    assert torch.equal(got, want)
    ctx2 = torch.randn(2, 77, 768, generator=g).to(DEV)
    runs = []
    for unet, c in ((four, None), (zeroed, cond[:1].to(DEV))):
        sch = _sched("ddim")[0]
        runs.append(denoise_loop(unet, sch, lat[:1].to(DEV), ctx2, 50, 7.5, cond=c))
        assert len(unet._samplers) == 1, "the run did not take the captured sampler"
    assert torch.equal(runs[1], runs[0])
    del zeroed, four
    torch.cuda.empty_cache()


@pytest.mark.parametrize("hw", [(64, 64), (96, 64)])
def test_full_size_forward_both_plans_vs_oracle(full, hw):
    oracle, ours = full
    h, w = hw
    g = torch.Generator().manual_seed(h)
    x = torch.cat([torch.randn(2, 4, h, w, generator=g), _cond(2, h, w, 5)], 1)
    ctx = torch.randn(2, 77, 768, generator=g)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = oc(x.to(DEV), 700, ctx.to(DEV)).sample.cpu()
    finally:
        oracle.to("cpu")
    rel = {}
    try:
        for prec in ("bf16", "fp32"):
            ours.set_precision(prec)
            with torch.no_grad():
                got = ours(x.to(DEV), 700, ctx.to(DEV)).sample.cpu()
            rel[prec] = float((got - want).abs().max() / want.abs().max())
    finally:
        ours.set_precision("bf16")
    print(f"9-channel UNet {h}x{w} batch 2: max-rel bf16 plan {rel['bf16']:.3g}, fp32 plan {rel['fp32']:.3g}")
    assert rel["bf16"] <= 1e-2 and rel["fp32"] <= 1e-4, rel


def _oracle_chain(oracle, kind, lat, cond, ctx2, n, dev, generator=None):
    _, ref, eta = _sched(kind)
    oc = oracle.to(dev)
    try:
        with torch.no_grad():
            return P9.denoise_loop(oc, ref, lat.to(dev), cond[:, :1].to(dev), cond[:, 1:].to(dev), ctx2.to(dev), n, 7.5, eta=eta,
                                   generator=generator).cpu()
    finally:
        oracle.to("cpu")


@pytest.mark.parametrize("kind", ["ddim", "plms"])
def test_captured_full_size_vs_oracle_and_per_call(full, kind):
    from b200sd.pipeline import denoise_loop
    oracle, ours = full
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    cond = _cond(1, 64, 64, 6)
    want = _oracle_chain(oracle, kind, lat, cond, ctx2, 50, DEV)
    ours.__dict__.pop("_samplers", None)
    got = denoise_loop(ours, _sched(kind)[0], lat.to(DEV), ctx2.to(DEV), 50, 7.5, cond=cond.to(DEV)).cpu()
    (smp,) = ours._samplers.values()
    assert smp.n_cond == 5 and tuple(smp.x2.shape) == (2, 9, 64, 64) and tuple(smp.latents.shape) == (1, 4, 64, 64)
    per_call = denoise_loop(ours, _sched(kind)[0], lat.to(DEV), ctx2.to(DEV), 50, 7.5, record=[], cond=cond.to(DEV)).cpu()
    cos, cos2 = _cos(got, want), _cos(got, per_call)
    print(f"{kind} 9-channel: captured vs fp32 oracle cosine {cos:.6f}, vs per-call {cos2:.6f}")
    assert cos >= 0.999 and cos2 >= 0.9999, (cos, cos2)


# ---------------------------------------------------------------------------------------------------
# every scheduler on the reduced-width net, batch 2, portrait latents
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    oracle = make_oracle_unet(seed=0, in_channels=9, **TINY_OVERRIDES)
    ours = UNet2DConditionModel(in_channels=9, **TINY_OVERRIDES)
    ours.load_state_dict(oracle.state_dict(), strict=True)
    return oracle, ours.to(DEV).eval()


def _tiny_inputs(seed=11):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(2, 4, 48, 32, generator=g), _cond(2, 48, 32, seed + 1), torch.randn(4, 77, 64, generator=g)


@pytest.mark.parametrize("kind", ["lms", "euler", "euler_ancestral"])
def test_sigma_schedulers_captured_equals_per_call_tiny_net(tiny, kind):
    """bit-identical to the per-call loop (the same kernels on the same values, concatenated then scaled as in 0.7.2), and the
    oracle chain with 0.7.2's order -- scaling the mask and the masked latents too -- within cosine 0.999"""
    from b200sd.pipeline import denoise_loop
    oracle, ours = tiny
    lat, cond, ctx2 = _tiny_inputs()
    gen = lambda: torch.Generator().manual_seed(0)
    want = _oracle_chain(oracle, kind, lat, cond, ctx2, 25, "cpu", generator=gen())
    ours.__dict__.pop("_samplers", None)
    got = denoise_loop(ours, _sched(kind)[0], lat.to(DEV), ctx2.to(DEV), 25, 7.5, generator=gen(), cond=cond.to(DEV)).cpu()
    assert len(ours._samplers) == 1
    per_call = denoise_loop(ours, _sched(kind)[0], lat.to(DEV), ctx2.to(DEV), 25, 7.5, record=[], generator=gen(),
                            cond=cond.to(DEV)).cpu()
    cos = _cos(got, want)
    print(f"{kind} 9-channel tiny: captured vs oracle cosine {cos:.6f}, bit-identical to per-call {torch.equal(got, per_call)}")
    assert torch.equal(got, per_call)
    assert cos >= 0.999, cos
    # the mask and the masked latents reach every step
    assert not torch.equal(got, denoise_loop(ours, _sched(kind)[0], lat.to(DEV), ctx2.to(DEV), 25, 7.5, generator=gen(),
                                             cond=(cond * 0.5).to(DEV)).cpu())


@pytest.mark.parametrize("kind", ["ddpm", "ddim_eta1"])
def test_stochastic_captured_reproduces_tiny_net(tiny, kind):
    from b200sd.pipeline import denoise_loop
    oracle, ours = tiny
    lat, cond, ctx2 = _tiny_inputs(seed=21)
    eta = _sched(kind)[2]
    run = lambda seed, **kw: denoise_loop(ours, _sched(kind)[0], lat.to(DEV), ctx2.to(DEV), 10, 7.5, eta=eta,
                                          generator=torch.Generator(DEV).manual_seed(seed), cond=cond.to(DEV), **kw).cpu()
    got = run(3)
    assert any(smp.noise.shape[0] > 0 for smp in ours._samplers.values())
    assert torch.equal(run(3), got), "the same generator seed must reproduce the run bit for bit"
    assert not torch.equal(run(4), got)
    cos = _cos(got, run(3, record=[]))
    print(f"{kind} 9-channel tiny: captured vs per-call cosine {cos:.6f}")
    assert cos >= 0.9999, cos


def test_kernels_per_step_against_text_to_image(tiny):
    """the input assembly is one counted launch: it replaces two torch copies (DDIM, PLMS, DDPM: one more kernel) or
    sampler_scale_input (the sigma schedulers: the same count)"""
    from b200sd.sampler import CapturedSampler
    from b200sd.unet import UNet2DConditionModel
    oracle, nine = tiny
    from oracle.unet_ref import TINY_OVERRIDES
    four = UNet2DConditionModel(**TINY_OVERRIDES)
    sd = {k: v.detach().cpu() for k, v in nine.state_dict().items()}
    sd["conv_in.weight"] = sd["conv_in.weight"][:, :4].clone()
    four.load_state_dict(sd, strict=True)
    four = four.to(DEV).eval()
    lat, cond, ctx2 = _tiny_inputs()
    counts = {}
    for kind in KINDS:
        row = []
        for unet, c in ((four, None), (nine, (cond[:, :1].to(DEV), cond[:, 1:].to(DEV)))):
            sch, _, eta = _sched(kind)
            sch.set_timesteps(6)
            smp = CapturedSampler(unet, sch, 2, 48, 32, 77, 7.5, eta=eta)
            smp.run(lat.to(DEV), ctx2.to(DEV), generator=torch.Generator().manual_seed(0), cond=c)
            row.append(smp.kernels_per_step)
        counts[kind] = tuple(row)
    print("kernels per step (text-to-image, 9-channel):", counts)
    for kind, (t2i, nine_ch) in counts.items():
        assert nine_ch == t2i + (0 if kind in ("lms", "euler", "euler_ancestral") else 1), (kind, t2i, nine_ch)


# ---------------------------------------------------------------------------------------------------
# the pipeline end to end on the reduced-width UNet and VAE
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny_pipe(tiny):
    from b200sd.vae import AutoencoderKL
    from oracle.vae_ref import TINY_VAE_OVERRIDES, make_oracle_vae
    o_vae = make_oracle_vae(seed=2, **TINY_VAE_OVERRIDES)
    vae = AutoencoderKL(**TINY_VAE_OVERRIDES)
    vae.load_state_dict(o_vae.state_dict(), strict=True)
    return tiny[0], o_vae, tiny[1], vae.to(DEV).eval()


def _pil_image(w, h):
    import numpy as np
    from PIL import Image
    yy, xx = np.mgrid[0:h, 0:w] / np.array([h, w]).reshape(2, 1, 1)
    arr = np.stack([0.5 + 0.4 * np.sin(2 * np.pi * (xx + 0.3 * yy)), 0.5 + 0.4 * np.cos(3 * np.pi * yy),
                    0.3 + 0.5 * xx * yy], -1)
    return Image.fromarray((arr * 255).round().astype(np.uint8), "RGB")


def _pil_mask(w, h):
    from PIL import Image
    m = Image.new("L", (w, h), 0)
    m.paste(255, (0, h // 4, w, h // 2))           # repaint the title band
    return m


@pytest.mark.parametrize("gen_device", ["cpu", "cuda"])
def test_pipeline_end_to_end_vs_oracle_chain(tiny_pipe, gen_device):
    """The whole chain (mask and masked image, the draws in 0.7.2's order -- initial latents, then the masked image's posterior
    sample --, bf16 VAE encode, the captured steps on [latents | mask | masked latents], VAE decode) against the fp32 oracle
    chain on the same draws.  Final latents: cosine >= 0.999.  Image: within 2e-2 max abs or the oracle chain's own error under
    torch's bf16 autocast, the yardstick of the legacy inpainting test."""
    from b200sd import StableDiffusionInpaintPipeline
    from b200sd.schedulers import DDIMScheduler
    o_unet, o_vae, unet, vae = tiny_pipe
    w, h = 256, 384
    pipe = StableDiffusionInpaintPipeline(vae=vae, unet=unet, scheduler=DDIMScheduler(**_DDIM_KW))
    ctx2 = torch.randn(4, 77, 64, generator=torch.Generator().manual_seed(5))
    image, mask = _pil_image(w, h), _pil_mask(w, h)
    mk = lambda: torch.Generator(gen_device).manual_seed(17)
    unet.__dict__.pop("_samplers", None)
    call = lambda output_type: pipe(prompt_embeds=ctx2.to(DEV), image=image, mask_image=mask, height=h, width=w,
                                    num_inference_steps=8, generator=mk(), output_type=output_type).images
    out, lat = call("pt"), call("latent")
    assert unet._samplers, "the pipeline did not sample on the captured graph"
    g = mk()                                          # the same draws, in the pipeline's order
    init = torch.randn((2, 4, h // 8, w // 8), generator=g, device=gen_device).cpu()
    post = torch.randn((1, 4, h // 8, w // 8), generator=g, device=gen_device).cpu()
    m, mi = P9.prepare_mask_and_masked_image(image, mask)
    args = lambda dev: (m.to(dev), mi.to(dev), ctx2.to(dev), 8, init.to(dev), post.to(dev))
    with torch.no_grad():
        want, want_lat = P9.pipeline(o_unet, o_vae, R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), *args("cpu"))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            lib, _ = P9.pipeline(copy.deepcopy(o_unet).to(DEV), copy.deepcopy(o_vae).to(DEV),
                                 R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), *args(DEV))
    assert tuple(out.shape) == (2, 3, h, w)
    err, err_lib = float((out.cpu() - want).abs().max()), float((lib.float().cpu() - want).abs().max())
    cos = _cos(lat, want_lat)
    print(f"9-channel inpaint {w}x{h} {gen_device} generator: image max abs {err:.4g} (torch bf16 autocast {err_lib:.4g}); "
          f"latents cosine {cos:.6f}")
    assert cos >= 0.999, cos
    assert err <= max(2e-2, err_lib), (err, err_lib)
