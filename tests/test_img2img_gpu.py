"""Image-to-image and legacy inpainting on the GPU: the masking kernel (inpaint_blend) against its fp32 formula and its table
form against its by-value form, runs that start at t_start on the captured sampler against the fp32 oracle
(oracle/img2img_ref.py) and the per-call loop, the exact properties of the mask, and the two pipelines end to end on the
reduced-width UNet and VAE."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

from oracle import ancestral_ref as A
from oracle import img2img_ref as I
from oracle import schedulers_ref as R

_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
_DDIM_KW = dict(_KW, clip_sample=False, set_alpha_to_one=False)


def _cos(a, b):
    return float(F.cosine_similarity(a.float().cpu().flatten(), b.float().cpu().flatten(), dim=0))


def _sched(kind):
    """(ours, oracle, eta)"""
    from b200sd.schedulers import DDIMScheduler, DDPMScheduler, PNDMScheduler
    if kind == "plms":
        return PNDMScheduler(**_KW, skip_prk_steps=True), R.PNDMSchedulerRef(skip_prk_steps=True), 0.0
    if kind == "ddpm":
        return DDPMScheduler(num_train_timesteps=1000, **_KW), A.DDPMSchedulerRef(), 0.0
    eta = 1.0 if kind == "ddim_eta1" else 0.0
    return DDIMScheduler(**_DDIM_KW), A.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), eta


# ---------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1, 4, 64, 64), (3, 4, 5, 7), (2, 4, 9, 9), (4, 4, 96, 64)])
def test_inpaint_blend_matches_fp32_formula(shape):
    from b200sd import ops
    from b200sd.schedulers import DDIMScheduler
    g = torch.Generator().manual_seed(shape[2])
    x, x0, z = (torch.randn(shape, generator=g) for _ in range(3))
    mask = torch.rand((shape[0], 1, shape[2], shape[3]), generator=g).expand(shape).contiguous()   # one mask per image
    mask[0] = 1.0
    sch = DDIMScheduler(**_DDIM_KW)
    sa, sb = sch._noise_tables(DEV)
    for t in (999, 501, 0, -3, 1200):
        tc = min(max(t, 0), 999)
        want = mask * (sa[tc].cpu() * x0 + sb[tc].cpu() * z) + (1 - mask) * x
        got = ops.inpaint_blend(x.to(DEV), x0.to(DEV), z.to(DEV), mask.to(DEV), t, sa, sb).cpu()
        torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-6 * float(want.abs().max()))
        noised = sch.add_noise(x0[:1].to(DEV), z[:1].to(DEV), torch.tensor([tc])).cpu()      # image 0 keeps everything
        torch.testing.assert_close(got[:1], noised, rtol=1e-6, atol=1e-6 * float(noised.abs().max()))


def test_inpaint_blend_table_equals_by_value_bit_for_bit():
    from b200sd import ops
    from b200sd.schedulers import DDIMScheduler
    sch = DDIMScheduler(**_DDIM_KW)
    sch.set_timesteps(50)
    sa, sb = sch._noise_tables(DEV)
    g = torch.Generator(DEV).manual_seed(2)
    shape = (2, 4, 64, 48)
    x, x0, z, m = (torch.randn(shape, generator=g, device=DEV) for _ in range(4))
    t_table = torch.tensor([float(t) for t in sch.timesteps.tolist()], device=DEV)
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    for k, t in enumerate(sch.timesteps.tolist()):
        want = ops.inpaint_blend(x.clone(), x0, z, m, t, sa, sb)
        cursor[1] = k
        got = ops.inpaint_blend_table(x.clone(), x0, z, m, t_table, cursor, sa, sb)
        assert torch.equal(got, want), f"step {k}"


# ---------------------------------------------------------------------------------------------------
# runs from t_start on the full-size SD v1.x network, latents given (no VAE)
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def models():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    oracle = make_oracle_unet(seed=0)
    ours = UNet2DConditionModel()
    ours.load_state_dict(oracle.state_dict(), strict=True)
    return oracle, ours.to(DEV).eval()


def _inputs(B=1, h=64, w=64, seed=42, ctx_dim=768):
    g = torch.Generator().manual_seed(seed)
    init = 0.8 * torch.randn(B, 4, h, w, generator=g)
    noise = torch.randn(B, 4, h, w, generator=g)
    ctx2 = torch.randn(2 * B, 77, ctx_dim, generator=g)
    return init, noise, ctx2


def _half_mask(B, h, w):
    m = torch.zeros(1, 4, h, w)
    m[:, :, : h // 2] = 1.0              # keep the top half, repaint the bottom
    return m.expand(B, 4, h, w)


def _ours(unet, sch, init, noise, ctx2, n, strength, mask=None, per_call=False, eta=0.0, generator=None):
    """ours from t_start: add_noise to t_noise, then denoise_loop (captured, or the per-call loop with per_call=True)"""
    from b200sd.pipeline import denoise_loop
    t_start, t_noise = sch.img2img_start(n, strength)
    lat = sch.add_noise(init.to(DEV), noise.to(DEV), torch.tensor([t_noise] * init.shape[0]))
    blend = None if mask is None else (init.to(DEV), noise.to(DEV), mask.to(DEV))
    return denoise_loop(unet, sch, lat, ctx2.to(DEV), n, 7.5, record=[] if per_call else None, eta=eta, generator=generator,
                        start=t_start, blend=blend)


@pytest.mark.parametrize("inpaint", [False, True])
@pytest.mark.parametrize("kind", ["ddim", "plms"])
def test_captured_from_t_start_vs_oracle_and_per_call(models, kind, inpaint):
    oracle, ours = models
    init, noise, ctx2 = _inputs()
    mask = _half_mask(1, 64, 64) if inpaint else None
    _, ref, _ = _sched(kind)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = I.denoise_loop(oc, ref, init.to(DEV), noise.to(DEV), ctx2.to(DEV), 50, 0.75,
                                  mask=None if mask is None else mask.to(DEV)).cpu()
    finally:
        oracle.to("cpu")
    ours.__dict__.pop("_samplers", None)
    got = _ours(ours, _sched(kind)[0], init, noise, ctx2, 50, 0.75, mask).cpu()
    (smp,) = ours._samplers.values()
    assert smp.n_steps == (38 if kind == "plms" else 37) and smp.inpaint == inpaint
    cos = _cos(got, want)
    print(f"{kind} inpaint={inpaint}: captured vs fp32 oracle cosine {cos:.6f}")
    assert cos >= 0.999, cos
    per_call = _ours(ours, _sched(kind)[0], init, noise, ctx2, 50, 0.75, mask, per_call=True).cpu()
    cos2 = _cos(got, per_call)
    print(f"{kind} inpaint={inpaint}: captured vs per-call cosine {cos2:.6f}")
    assert cos2 >= 0.9999, cos2


def test_mask_exact_properties_and_launch_counts(models):
    from b200sd.sampler import CapturedSampler
    _, ours = models
    init, noise, ctx2 = _inputs(seed=7)
    sch = _sched("ddim")[0]
    img2img = _ours(ours, sch, init, noise, ctx2, 50, 0.75).cpu()
    repaint_all = _ours(ours, sch, init, noise, ctx2, 50, 0.75, mask=torch.zeros(1, 4, 64, 64)).cpu()
    assert torch.equal(repaint_all, img2img), "an all-zero keep-mask must leave img2img unchanged"
    keep_all = _ours(ours, sch, init, noise, ctx2, 50, 0.75, mask=torch.ones(1, 4, 64, 64))
    t_last = int(sch.timesteps[-1])
    want = sch.add_noise(init.to(DEV), noise.to(DEV), torch.tensor([t_last]))
    torch.testing.assert_close(keep_all, want, rtol=1e-6, atol=1e-6 * float(want.abs().max()))
    counts = {}
    for name, start, inpaint in (("t2i", 0, False), ("img2img", 13, False), ("inpaint", 13, True)):
        sch.set_timesteps(50)
        smp = CapturedSampler(ours, sch, 1, 64, 64, 77, 7.5, start=start, inpaint=inpaint)
        blend = (init, noise, torch.ones(1, 4, 64, 64)) if inpaint else None
        smp.run(init.to(DEV), ctx2.to(DEV), blend=blend)
        counts[name] = smp.kernels_per_step
    print("kernels per step", counts)
    assert counts["img2img"] == counts["t2i"] > 0 and counts["inpaint"] == counts["t2i"] + 1


# ---------------------------------------------------------------------------------------------------
# stochastic samplers on the reduced-width network
# ---------------------------------------------------------------------------------------------------
def _tiny_unet():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    unet = UNet2DConditionModel(**TINY_OVERRIDES)
    unet.load_state_dict(make_oracle_unet(seed=0, **TINY_OVERRIDES).state_dict(), strict=True)
    return unet.to(DEV).eval()


@pytest.mark.parametrize("inpaint", [False, True])
@pytest.mark.parametrize("kind", ["ddpm", "ddim_eta1"])
def test_stochastic_captured_vs_per_call_tiny_net(kind, inpaint):
    unet = _tiny_unet()
    init, noise, ctx2 = _inputs(B=2, h=32, w=32, seed=11, ctx_dim=64)
    mask = _half_mask(2, 32, 32) if inpaint else None
    eta = _sched(kind)[2]
    gen = lambda: torch.Generator(DEV).manual_seed(3)
    got = _ours(unet, _sched(kind)[0], init, noise, ctx2, 10, 0.75, mask, eta=eta, generator=gen())
    assert any(smp.noise.shape[0] > 0 for smp in unet._samplers.values())
    again = _ours(unet, _sched(kind)[0], init, noise, ctx2, 10, 0.75, mask, eta=eta, generator=gen())
    assert torch.equal(got, again), "the same generator seed must reproduce the run bit for bit"
    per_call = _ours(unet, _sched(kind)[0], init, noise, ctx2, 10, 0.75, mask, per_call=True, eta=eta, generator=gen())
    cos = _cos(got, per_call)
    assert cos >= 0.9999, cos


# ---------------------------------------------------------------------------------------------------
# the pipelines end to end on the reduced-width UNet and VAE
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny():
    from b200sd.vae import AutoencoderKL
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    from oracle.vae_ref import TINY_VAE_OVERRIDES, make_oracle_vae
    o_unet, o_vae = make_oracle_unet(seed=0, **TINY_OVERRIDES), make_oracle_vae(seed=2, **TINY_VAE_OVERRIDES)
    vae = AutoencoderKL(**TINY_VAE_OVERRIDES)
    vae.load_state_dict(o_vae.state_dict(), strict=True)
    return o_unet, o_vae, _tiny_unet(), vae.to(DEV).eval()


def _pil_image(w, h):
    """a smooth picture, like a layout sketch or a cover"""
    import numpy as np
    from PIL import Image
    yy, xx = np.mgrid[0:h, 0:w] / np.array([h, w]).reshape(2, 1, 1)
    arr = np.stack([0.5 + 0.4 * np.sin(2 * np.pi * (xx + 0.3 * yy)), 0.5 + 0.4 * np.cos(3 * np.pi * yy),
                    0.3 + 0.5 * xx * yy], -1)
    return Image.fromarray((arr * 255).round().astype(np.uint8), "RGB")


def _pil_mask(w, h):
    from PIL import Image
    m = Image.new("L", (w, h), 0)
    m.paste(255, (0, h // 4, w, h // 2))           # repaint a band, as for a title
    return m


@pytest.mark.parametrize("gen_device", ["cpu", "cuda"])
@pytest.mark.parametrize("w,h", [(256, 256), (256, 384)])
@pytest.mark.parametrize("inpaint", [False, True])
def test_pipeline_end_to_end_vs_oracle_chain(tiny, inpaint, w, h, gen_device):
    """The whole chain (preprocess, bf16 VAE encode, posterior sample, add_noise, the steps from t_start, the masking step, VAE
    decode) against the fp32 oracle chain on the same draws.  The final latents must agree (cosine >= 0.999).  The image must be
    within 2e-2 max abs, or not worse than the oracle chain itself under torch's bf16 autocast: the bf16 VAE alone, encoding
    and decoding the image, reaches ~2e-2 here (the kept region of the inpainting runs is exactly that), so the image bar
    follows tests/test_vae_gpu.py's library-bf16 yardstick."""
    from b200sd import StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy
    from b200sd.schedulers import DDIMScheduler
    o_unet, o_vae, unet, vae = tiny
    cls = StableDiffusionInpaintPipelineLegacy if inpaint else StableDiffusionImg2ImgPipeline
    pipe = cls(vae=vae, unet=unet, scheduler=DDIMScheduler(**_DDIM_KW))
    ctx2 = torch.randn(4, 77, 64, generator=torch.Generator().manual_seed(5))
    image, mask = _pil_image(w, h), _pil_mask(w, h)
    kw = dict(mask_image=mask) if inpaint else {}
    mk = lambda: torch.Generator(gen_device).manual_seed(17)
    unet.__dict__.pop("_samplers", None)
    call = lambda output_type: pipe(prompt_embeds=ctx2.to(DEV), init_image=image, strength=0.75, num_inference_steps=8,
                                    generator=mk(), output_type=output_type, **kw).images
    out, lat = call("pt"), call("latent")
    assert unet._samplers, "the pipeline did not sample on the captured graph"
    g = mk()                                          # the same draws, in the pipeline's order
    post_noise = torch.randn((1, 4, h // 8, w // 8), generator=g, device=gen_device).cpu()
    init_noise = torch.randn((2, 4, h // 8, w // 8), generator=g, device=gen_device).cpu()
    ref_args = lambda dev: (I.preprocess_image(image).to(dev), ctx2.to(dev), 8, 0.75, post_noise.to(dev), init_noise.to(dev))
    ref_mask = lambda dev: I.preprocess_mask(mask).to(dev) if inpaint else None
    with torch.no_grad():
        want, want_lat = I.pipeline(o_unet, o_vae, R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), *ref_args("cpu"),
                                    mask=ref_mask("cpu"))
        # the library bf16 yardstick of tests/test_vae_gpu.py: the same oracle chain under torch's bf16 autocast, same draws
        with torch.autocast("cuda", dtype=torch.bfloat16):
            lib, _ = I.pipeline(copy.deepcopy(o_unet).to(DEV), copy.deepcopy(o_vae).to(DEV),
                                R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), *ref_args(DEV), mask=ref_mask(DEV))
    assert tuple(out.shape) == (2, 3, h, w)
    err, err_lib = float((out.cpu() - want).abs().max()), float((lib.float().cpu() - want).abs().max())
    cos = _cos(lat, want_lat)
    print(f"inpaint={inpaint} {w}x{h} {gen_device} generator: image max abs {err:.4g} (torch bf16 autocast {err_lib:.4g}); "
          f"latents cosine {cos:.6f}")
    assert cos >= 0.999, cos
    assert err <= max(2e-2, err_lib), (err, err_lib)


def test_saved_pipeline_samples_in_both_classes_and_text_to_image_still_matches(tiny, tmp_path):
    from b200sd import StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy, StableDiffusionPipeline
    from b200sd.schedulers import DDIMScheduler
    _, _, unet, vae = tiny
    StableDiffusionPipeline(vae=vae, unet=unet, scheduler=DDIMScheduler(**_DDIM_KW)).save_pretrained(str(tmp_path))
    ctx2 = torch.randn(2, 77, 64, generator=torch.Generator().manual_seed(8)).to(DEV)
    lat = torch.randn(1, 4, 32, 32, generator=torch.Generator().manual_seed(9)).to(DEV)
    t2i = StableDiffusionPipeline.from_pretrained(str(tmp_path)).to(DEV)
    fresh = t2i(prompt_embeds=ctx2, height=256, width=256, num_inference_steps=6, latents=lat, output_type="latent").images
    image = torch.rand(1, 3, 256, 256, generator=torch.Generator().manual_seed(1)) * 2 - 1
    for cls, kw in ((StableDiffusionImg2ImgPipeline, {}),
                    (StableDiffusionInpaintPipelineLegacy, dict(mask_image=torch.ones(1, 4, 32, 32) * 0.5))):
        pipe = cls.from_pretrained(str(tmp_path)).to(DEV)
        out = pipe(prompt_embeds=ctx2, init_image=image, strength=0.5, num_inference_steps=6, output_type="pt",
                   generator=torch.Generator().manual_seed(0), **kw).images
        assert tuple(out.shape) == (1, 3, 256, 256) and bool(torch.isfinite(out).all())
    # the same UNet object now also holds samplers that start at t_start: text-to-image must not pick one up
    t2i.unet = pipe.unet
    assert any(key[-2] > 0 for key in pipe.unet._samplers)
    again = t2i(prompt_embeds=ctx2, height=256, width=256, num_inference_steps=6, latents=lat, output_type="latent").images
    assert torch.equal(again, fresh)
