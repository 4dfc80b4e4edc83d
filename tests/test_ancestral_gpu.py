"""Ancestral sampling on the GPU (DDPMScheduler; DDIMScheduler with eta > 0): the fused step kernel against the fp32 oracle
restatement of diffusers 0.7.2, its table form against the per-call form bit for bit, the facade loops, the captured sampler
on the full-size and the reduced-width network, and StableDiffusionPipeline.__call__ with a saved DDPMScheduler."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

from oracle import ancestral_ref as A
from oracle import schedulers_ref as R

_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
_DDIM_KW = dict(_KW, clip_sample=False, set_alpha_to_one=False)


def _cos(a, b):
    return float(F.cosine_similarity(a.float().cpu().flatten(), b.float().cpu().flatten(), dim=0))


def _pair(kind, n=50):
    """(ours, oracle, eta) with set_timesteps(n) done"""
    from b200sd.schedulers import DDIMScheduler, DDPMScheduler
    if kind == "ddpm":
        ours, ref, eta = DDPMScheduler(num_train_timesteps=1000, **_KW), A.DDPMSchedulerRef(), 0.0
    else:
        ours, ref, eta = DDIMScheduler(**_DDIM_KW), A.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), 1.0
    ours.set_timesteps(n)
    ref.set_timesteps(n)
    return ours, ref, eta


def _ref_step(ref, eta, eps, t, x, g):
    return ref.step(eps, t, x, generator=g) if eta == 0.0 else ref.step(eps, t, x, eta=eta, generator=g)


@pytest.mark.parametrize("n_shape", [(1, 4, 64, 64), (3, 4, 96, 64), (1, 4, 5, 7), (2, 3, 1, 1)])
@pytest.mark.parametrize("cfg", [True, False])
@pytest.mark.parametrize("eps_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("kind", ["ddpm", "ddim_eta1"])
def test_cfg_ancestral_step_vs_oracle(n_shape, cfg, eps_dtype, kind):
    from b200sd import ops
    from b200sd.schedulers import step_noise
    torch.manual_seed(0)
    B = n_shape[0]
    x = torch.randn(n_shape)
    eps2 = torch.randn((2 * B if cfg else B,) + n_shape[1:]).to(eps_dtype)
    ours, ref, eta = _pair(kind)
    for t in (980, 500, 1, 0):
        eps = R.cfg_combine(eps2.float(), 7.5) if cfg else eps2.float()
        want = _ref_step(ref, eta, eps, t, x, torch.Generator().manual_seed(t)).prev_sample
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noisy, clip = ours._ancestral_coefs(t, eta)
        z = step_noise(x.to(DEV), torch.Generator().manual_seed(t)) if noisy else None
        e2 = eps2.to(DEV)
        eu, ec = (e2[:B].contiguous(), e2[B:].contiguous()) if cfg else (e2, None)
        got = ops.cfg_ancestral_step(eu, ec, x.to(DEV), z, 7.5, sa_t, sb_t, c_x0, c_x, c_e, c_z, clip)
        torch.testing.assert_close(got.cpu(), want, rtol=2e-6, atol=2e-6 * float(want.abs().max()))


@pytest.mark.parametrize("kind", ["ddpm", "ddim_eta1"])
def test_table_kernel_equals_per_call_kernel_bit_for_bit(kind):
    from b200sd import ops
    ours, _ref, eta = _pair(kind)
    rows, n_noisy = ours.ancestral_plan(eta)
    table = torch.tensor(rows, dtype=torch.float32, device=DEV)
    g = torch.Generator(DEV).manual_seed(1)
    shape = (2, 4, 64, 64)
    n = 2 * 4 * 64 * 64
    eu, ec, x = (torch.randn(shape, generator=g, device=DEV) for _ in range(3))
    noise = torch.randn(n_noisy, n, generator=g, device=DEV)
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    for k, row in enumerate(table.tolist()):
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noise_row, clip = row
        z = None if noise_row < 0 else noise[int(noise_row)].view(shape)
        want = ops.cfg_ancestral_step(eu, ec, x, z, 7.5, sa_t, sb_t, c_x0, c_x, c_e, c_z, clip != 0.0)
        cursor[1] = k
        got = x.clone()
        ops.cfg_ancestral_step_table(eu, ec, got, noise, 7.5, table, cursor)
        assert torch.equal(got, want), f"row {k}"


@pytest.mark.parametrize("kind", ["ddpm", "ddim_eta1"])
def test_facade_loop_matches_oracle(kind):
    torch.manual_seed(3)
    x = torch.randn(1, 4, 64, 64)
    ours, ref, eta = _pair(kind)
    assert ours.timesteps.tolist() == ref.timesteps.tolist()
    g_ref, g_ours = torch.Generator().manual_seed(9), torch.Generator().manual_seed(9)
    xr, xo = x.clone(), x.to(DEV)
    for i, t in enumerate(ref.timesteps):
        eps = torch.randn(x.shape, generator=torch.Generator().manual_seed(i))
        xr = _ref_step(ref, eta, eps, t, xr, g_ref).prev_sample
        if eta == 0.0:
            xo = ours.step(eps.to(DEV), t, xo, generator=g_ours).prev_sample
        else:
            xo = ours.step(eps.to(DEV), t, xo, eta=eta, generator=g_ours).prev_sample
    torch.testing.assert_close(xo.cpu(), xr, rtol=1e-5, atol=1e-5 * float(xr.abs().max()))


# ---------------------------------------------------------------------------------------------------
# the captured sampler on the full-size SD v1.x network
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


@pytest.mark.parametrize("kind", ["ddpm", "ddim_eta1"])
def test_captured_sampler_50_steps(models, kind):
    from b200sd.pipeline import denoise_loop
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    oracle, ours = models
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    _, ref, eta = _pair(kind)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = A.denoise_loop(oc, ref, lat.to(DEV), ctx2.to(DEV), 50, 7.5, eta=eta,
                                  generator=torch.Generator().manual_seed(0)).cpu()
    finally:
        oracle.to("cpu")
    sch, _, _ = _pair(kind)
    smp = CapturedSampler(ours, sch, 1, 64, 64, 77, 7.5, eta=eta)
    assert smp.noise.shape == (49 if kind == "ddpm" else 50, 4 * 64 * 64)
    got = smp.run(lat.to(DEV), ctx2.to(DEV), generator=torch.Generator().manual_seed(0)).cpu()
    cos = _cos(got, want)
    print(f"{kind}: captured vs fp32 oracle loop cosine {cos:.6f}")
    assert cos >= 0.999, f"{kind}: 50-step latents cosine {cos:.6f}"
    again = smp.run(lat.to(DEV), ctx2.to(DEV), generator=torch.Generator().manual_seed(0)).cpu()
    assert torch.equal(again, got), "the same generator seed must reproduce the run bit for bit"
    other = smp.run(lat.to(DEV), ctx2.to(DEV), generator=torch.Generator().manual_seed(1)).cpu()
    assert not torch.equal(other, got)
    sch2, _, _ = _pair(kind)
    per_call = denoise_loop(ours, sch2, lat.to(DEV), ctx2.to(DEV), 50, 7.5, record=[], eta=eta,
                            generator=torch.Generator().manual_seed(0)).cpu()
    cos2 = _cos(got, per_call)
    print(f"{kind}: captured vs per-call loop cosine {cos2:.6f}")
    assert cos2 >= 0.9999, f"{kind}: captured vs per-call cosine {cos2:.6f}"
    ddim = DDIMScheduler(**_DDIM_KW)
    ddim.set_timesteps(2)
    ref_smp = CapturedSampler(ours, ddim, 1, 64, 64, 77, 7.5)
    ref_smp.run(lat.to(DEV), ctx2.to(DEV))
    assert smp.kernels_per_step == ref_smp.kernels_per_step > 0


def test_captured_ddpm_batched_portrait_tiny_net():
    from b200sd.sampler import CapturedSampler
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    oracle = make_oracle_unet(seed=0, **TINY_OVERRIDES)
    ours = UNet2DConditionModel(**TINY_OVERRIDES)
    ours.load_state_dict(oracle.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(2, 4, 48, 32, generator=g)
    ctx2 = torch.randn(4, 77, 64, generator=g)
    sch, ref, _ = _pair("ddpm", 6)
    with torch.no_grad():
        want = A.denoise_loop(oracle, ref, lat, ctx2, 6, 7.5, generator=torch.Generator().manual_seed(5))
    got = CapturedSampler(ours, sch, 2, 48, 32, 77, 7.5, lanes=1).run(lat.to(DEV), ctx2.to(DEV),
                                                                       generator=torch.Generator().manual_seed(5)).cpu()
    cos = _cos(got, want)
    assert cos >= 0.999, f"cosine {cos:.6f}"


# ---------------------------------------------------------------------------------------------------
# StableDiffusionPipeline: what finetune_sd.py saves (a DDPMScheduler) samples on the captured graph
# ---------------------------------------------------------------------------------------------------
def _tiny_unet():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    unet = UNet2DConditionModel(**TINY_OVERRIDES)
    unet.load_state_dict(make_oracle_unet(seed=0, **TINY_OVERRIDES).state_dict(), strict=True)
    return unet


def _per_call(unet, scheduler, ctx2, generator, eta=0.0):
    """the pipeline's draws by hand: initial latents first, then the step noise, on the per-call loop"""
    from b200sd.pipeline import denoise_loop
    dev = "cpu" if generator.device.type == "cpu" else DEV
    lat = torch.randn((ctx2.shape[0] // 2, 4, 32, 32), generator=generator, device=dev).to(DEV)
    return denoise_loop(unet, scheduler, lat, ctx2, 6, 7.5, record=[], eta=eta, generator=generator)


def test_pipeline_saved_with_ddpm_samples_on_the_captured_graph(tmp_path):
    from b200sd import StableDiffusionPipeline
    from b200sd.schedulers import DDPMScheduler
    StableDiffusionPipeline(unet=_tiny_unet(), scheduler=DDPMScheduler(num_train_timesteps=1000, **_KW)).save_pretrained(
        str(tmp_path))
    pipe = StableDiffusionPipeline.from_pretrained(str(tmp_path)).to(DEV)
    assert isinstance(pipe.scheduler, DDPMScheduler)
    ctx2 = torch.randn(4, 77, 64, generator=torch.Generator().manual_seed(4)).to(DEV)
    for gen in (lambda: torch.Generator("cuda").manual_seed(0), lambda: torch.Generator().manual_seed(0)):
        pipe.unet.__dict__.pop("_samplers", None)
        out = pipe(prompt_embeds=ctx2, height=256, width=256, num_inference_steps=6, guidance_scale=7.5, generator=gen(),
                   output_type="latent")
        assert pipe.unet._samplers, "the pipeline did not sample on the captured graph"
        want = _per_call(pipe.unet, DDPMScheduler(num_train_timesteps=1000, **_KW), ctx2, gen())
        cos = _cos(out.images, want)
        assert out.images.shape == (2, 4, 32, 32) and cos >= 0.9999, cos


def test_pipeline_ddim_eta1(tmp_path):
    from b200sd import StableDiffusionPipeline
    from b200sd.schedulers import DDIMScheduler
    pipe = StableDiffusionPipeline(unet=_tiny_unet().eval(), scheduler=DDIMScheduler(**_DDIM_KW)).to(DEV)
    ctx2 = torch.randn(4, 77, 64, generator=torch.Generator().manual_seed(4)).to(DEV)
    out = pipe(prompt_embeds=ctx2, height=256, width=256, num_inference_steps=6, guidance_scale=7.5, eta=1.0,
               generator=torch.Generator("cuda").manual_seed(0), output_type="latent")
    assert any(smp.noise.shape[0] > 0 for smp in pipe.unet._samplers.values())
    want = _per_call(pipe.unet, DDIMScheduler(**_DDIM_KW), ctx2, torch.Generator("cuda").manual_seed(0), eta=1.0)
    cos = _cos(out.images, want)
    assert cos >= 0.9999, cos
    det = pipe(prompt_embeds=ctx2, height=256, width=256, num_inference_steps=6, guidance_scale=7.5,
               generator=torch.Generator("cuda").manual_seed(0), output_type="latent")
    assert not torch.equal(det.images, out.images), "eta = 1 must differ from the deterministic eta = 0 run"
