"""The sigma-space schedulers on the GPU (LMSDiscreteScheduler, EulerDiscreteScheduler, EulerAncestralDiscreteScheduler): the
fused step kernel against the fp32 oracle restatement of diffusers 0.7.2, its table form and the model-input scaling kernel
against the per-call forms bit for bit, diffusers' published full-loop answers, the UNet at a fractional timestep, the captured
sampler against the per-call loop and the oracle chain, and StableDiffusionPipeline loading and sampling each scheduler."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

from oracle import schedulers_ref as R
from oracle import sigma_ref as S

HERE = os.path.dirname(os.path.abspath(__file__))
KAT = json.load(open(os.path.join(HERE, "golden", "diffusers_0_7_2_sigma_kat.json")))
_SD = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
KINDS = ("lms", "euler", "euler_ancestral")


def _cos(a, b):
    return float(F.cosine_similarity(a.float().cpu().flatten(), b.float().cpu().flatten(), dim=0))


def _classes(kind):
    from b200sd import schedulers as B
    return {"lms": (B.LMSDiscreteScheduler, S.LMSDiscreteSchedulerRef),
            "euler": (B.EulerDiscreteScheduler, S.EulerDiscreteSchedulerRef),
            "euler_ancestral": (B.EulerAncestralDiscreteScheduler, S.EulerAncestralDiscreteSchedulerRef)}[kind]


def _pair(kind, n=50, **cfg):
    ours_cls, ref_cls = _classes(kind)
    cfg = cfg or _SD
    ours, ref = ours_cls(**cfg), ref_cls(**cfg)
    ours.set_timesteps(n)
    ref.set_timesteps(n)
    return ours, ref


def _gen_kw(kind, seed):
    return {"generator": torch.Generator().manual_seed(seed)} if kind == "euler_ancestral" else {}


# ---------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_shape", [(1, 4, 64, 64), (3, 4, 96, 64), (1, 4, 5, 7), (2, 3, 1, 1)])
@pytest.mark.parametrize("cfg", [True, False])
@pytest.mark.parametrize("eps_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("kind", KINDS)
def test_cfg_sigma_step_vs_oracle(n_shape, cfg, eps_dtype, kind):
    """A run of steps (the first five, so LMS reaches order 4, and the last) on the per-call path: the by-value entry point with
    its history pointers and derivative output, against the oracle on the CPU."""
    torch.manual_seed(0)
    B = n_shape[0]
    x = torch.randn(n_shape) * 10
    ours, ref = _pair(kind)
    xo, xr = x.to(DEV), x.clone()
    steps = list(range(5)) + [49]
    for i in steps:
        if i == 49:        # jump to the last step: both sides restart their LMS history there
            ours._derivs, ref.derivatives = [], []
        t = ref.timesteps[i]
        eps2 = torch.randn((2 * B if cfg else B,) + n_shape[1:]).to(eps_dtype)
        eps = R.cfg_combine(eps2.float(), 7.5) if cfg else eps2.float()
        want = ref.step(eps, t, xr, **_gen_kw(kind, i)).prev_sample
        e2 = eps2.to(DEV)
        if cfg:
            got = ours.step_cfg(e2, float(t), xo, 7.5, **_gen_kw(kind, i)).prev_sample
        else:
            got = ours.step(e2, float(t), xo, **_gen_kw(kind, i)).prev_sample
        torch.testing.assert_close(got.cpu(), want, rtol=2e-6, atol=2e-6 * float(want.abs().max()))
        xo, xr = got, want


@pytest.mark.parametrize("kind", KINDS)
def test_table_kernel_equals_per_call_kernel_bit_for_bit(kind):
    from b200sd import ops
    ours, _ = _pair(kind)
    rows, n_noise = ours.sigma_plan()
    table = torch.tensor(rows, dtype=torch.float32, device=DEV)
    g = torch.Generator(DEV).manual_seed(1)
    shape = (2, 4, 64, 64)
    n = 2 * 4 * 64 * 64
    eu, ec = (torch.randn(shape, generator=g, device=DEV) for _ in range(2))
    x = torch.randn(shape, generator=g, device=DEV) * 10
    noise = torch.randn(n_noise, n, generator=g, device=DEV) if n_noise else None
    ring = torch.randn(4, n, generator=g, device=DEV) if kind == "lms" else None
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    for k, row in enumerate(table.tolist()):
        sigma, c = row[0], row[1:5]
        hist = [ring[int(s)].view(shape) for s in row[5:8] if s >= 0]
        slot, noise_row, sigma_up = int(row[8]), int(row[9]), row[10]
        d = torch.empty_like(x) if slot >= 0 else None
        z = noise[noise_row].view(shape) if noise_row >= 0 else None
        want = ops.cfg_sigma_step(eu, ec, x, 7.5, sigma, c[:len(hist) + 1], hist, z, sigma_up, d_out=d)
        cursor[1] = k
        got, got_ring = x.clone(), None if ring is None else ring.clone()
        ops.cfg_sigma_step_table(eu, ec, got, got_ring, noise, 7.5, table, cursor)
        assert torch.equal(got, want), f"row {k}"
        if slot >= 0:
            assert torch.equal(got_ring[slot].view(shape), d), f"row {k}: derivative"
            ring = got_ring
        x = want


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", [(1, 4, 64, 64), (1, 3, 5, 7)])
def test_sampler_scale_input_equals_scale_model_input_bit_for_bit(kind, shape):
    from b200sd import ops
    ours, _ = _pair(kind)
    table = torch.tensor(ours.sigma_plan()[0], dtype=torch.float32, device=DEV)
    x = torch.randn(shape, device=DEV) * 14
    x2 = torch.empty((2 * shape[0],) + shape[1:], device=DEV)
    cursor = torch.zeros(2, dtype=torch.int32, device=DEV)
    for k, t in enumerate(ours.timesteps.tolist()):
        cursor[1] = k
        ops.sampler_scale_input(x, x2, table, cursor)
        want = ours.scale_model_input(torch.cat([x, x]), t)
        assert torch.equal(x2, want), f"step {k}"


@pytest.mark.parametrize("kind", KINDS)
def test_published_full_loop_on_the_kernels(kind):
    """diffusers 0.7.2's test_full_loop_no_noise with the facade's CUDA step (tests/golden/diffusers_0_7_2_sigma_kat.json)"""
    ours = _classes(kind)[0](num_train_timesteps=1100, beta_start=0.0001, beta_end=0.02, beta_schedule="linear")
    kw = {"generator": torch.manual_seed(0)} if kind == "euler_ancestral" else {}
    sample = kat_full_loop(ours, dict(kw, device=DEV)).cpu()
    want_sum, want_mean = KAT[kind]
    assert abs(float(sample.abs().sum()) - want_sum) < KAT["tolerances"]["sum_atol"]
    assert abs(float(sample.abs().mean()) - want_mean) < KAT["tolerances"]["mean_atol"]


def dummy_sample_deter():
    n = 4 * 3 * 8 * 8
    return (torch.arange(n).reshape(3, 8, 8, 4) / n).permute(3, 0, 1, 2)


def dummy_model(sample, t):
    return sample * t / (t + 1)


def kat_full_loop(sch, step_kw):
    """diffusers' test_full_loop_no_noise, including its overwrite of `sample` by scale_model_input"""
    sch.set_timesteps(10)
    sample = dummy_sample_deter().to(step_kw.pop("device", "cpu")) * sch.init_noise_sigma
    for t in sch.timesteps:
        sample = sch.scale_model_input(sample, t)
        sample = sch.step(dummy_model(sample, t), t, sample, **step_kw).prev_sample
    return sample


# ---------------------------------------------------------------------------------------------------
# the UNet at a fractional timestep
# ---------------------------------------------------------------------------------------------------
def test_timestep_embedding_fractional_t():
    from b200sd import ops
    from oracle.unet_ref import timestep_embedding
    ours, _ = _pair("lms")
    t = ours.timesteps[:6].to(torch.float32)
    assert any(float(v) != int(v) for v in t)
    got = ops.timestep_embedding(t.to(DEV), 320).cpu()
    want = timestep_embedding(ours.timesteps[:6], 320)       # float64 t, cast to fp32 inside, as 0.7.2's UNet does
    torch.testing.assert_close(got, want, rtol=0, atol=2e-4)  # the bar of the integer-t test: fp32 sin/cos of ~1e3 rad


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


def test_unet_forward_at_fractional_t(models):
    oracle, ours = models
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 64, 64, generator=g)
    ctx = torch.randn(1, 77, 768, generator=g)
    t = torch.tensor(978.6122448979592, dtype=torch.float64)    # timesteps[1] of a 50-step LMS / Euler schedule
    with torch.no_grad():
        want = oracle(x, t, ctx).sample
        got = ours(x.to(DEV), t, ctx.to(DEV)).sample.cpu()
        other = oracle(x, torch.tensor(978.0, dtype=torch.float64), ctx).sample
    r = float((got - want).abs().max() / want.abs().max())
    assert r <= 1e-2, f"max-rel {r:.4g}"
    assert not torch.equal(want, other), "the fraction must reach the embedding"


# ---------------------------------------------------------------------------------------------------
# the captured sampler
# ---------------------------------------------------------------------------------------------------
def _check_captured(oracle, ours, kind, B, h, w, S_ctx, ctx_dim, n, oracle_dev):
    from b200sd.pipeline import denoise_loop
    from b200sd.sampler import CapturedSampler
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(B, 4, h, w, generator=g)
    ctx2 = torch.randn(2 * B, S_ctx, ctx_dim, generator=g)
    _, ref = _pair(kind, n)
    oc = oracle.to(oracle_dev)
    try:
        with torch.no_grad():
            want = S.denoise_loop(oc, ref, lat.to(oracle_dev), ctx2.to(oracle_dev), n, 7.5,
                                  generator=torch.Generator().manual_seed(0)).cpu()
    finally:
        oracle.to("cpu")
    sch, _ = _pair(kind, n)
    smp = CapturedSampler(ours, sch, B, h, w, S_ctx, 7.5)
    assert smp.noise.shape[0] == (n if kind == "euler_ancestral" else 0)
    assert smp.ring.shape[0] == (4 if kind == "lms" else 0)
    got = smp.run(lat.to(DEV), ctx2.to(DEV), generator=torch.Generator().manual_seed(0)).cpu()
    cos = _cos(got, want)
    print(f"{kind}: captured vs fp32 oracle loop cosine {cos:.6f}")
    assert cos >= 0.999, f"{kind}: {n}-step latents cosine {cos:.6f}"
    sch2, _ = _pair(kind, n)
    per_call = denoise_loop(ours, sch2, lat.to(DEV), ctx2.to(DEV), n, 7.5, record=[],
                            generator=torch.Generator().manual_seed(0)).cpu()
    cos2 = _cos(got, per_call)
    print(f"{kind}: captured vs per-call loop cosine {cos2:.6f}, bit-identical {torch.equal(got, per_call)}")
    assert cos2 >= 0.9999, f"{kind}: captured vs per-call cosine {cos2:.6f}"
    return smp, got, per_call, lat, ctx2


def test_captured_lms_50_steps_full_size(models):
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    oracle, ours = models
    smp, got, _, lat, ctx2 = _check_captured(oracle, ours, "lms", 1, 64, 64, 77, 768, 50, DEV)
    again = smp.run(lat.to(DEV), ctx2.to(DEV)).cpu()
    assert torch.equal(again, got), "a second run must reproduce the first bit for bit (the ring is rewritten before it is read)"
    ddim = DDIMScheduler(**_SD, clip_sample=False, set_alpha_to_one=False)
    ddim.set_timesteps(2)
    ref_smp = CapturedSampler(ours, ddim, 1, 64, 64, 77, 7.5)
    ref_smp.run(lat.to(DEV), ctx2.to(DEV))
    # sampler_scale_input replaces the two latents copies (torch copies, not counted), so one more counted launch
    assert smp.kernels_per_step == ref_smp.kernels_per_step + 1


@pytest.fixture(scope="module")
def tiny():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    oracle = make_oracle_unet(seed=0, **TINY_OVERRIDES)
    ours = UNet2DConditionModel(**TINY_OVERRIDES)
    ours.load_state_dict(oracle.state_dict(), strict=True)
    return oracle, ours.to(DEV).eval()


@pytest.mark.parametrize("kind", ["euler", "euler_ancestral"])
def test_captured_euler_batched_portrait_tiny_net(tiny, kind):
    oracle, ours = tiny
    smp, got, per_call, lat, ctx2 = _check_captured(oracle, ours, kind, 2, 48, 32, 77, 64, 25, "cpu")
    if kind == "euler_ancestral":
        # the same generator gives the same latents on both loops: the captured run's noise table holds exactly the per-call
        # loop's draws, in step order, and both run the same kernels on the same values
        assert torch.equal(got, per_call)
        g = torch.Generator().manual_seed(0)
        from b200sd.schedulers import step_noise
        for k in range(smp.noise.shape[0]):
            z = step_noise(smp.latents, g)
            assert torch.equal(smp.noise[k].view(z.shape), z), f"noise row {k}"
        other = smp.run(lat.to(DEV), ctx2.to(DEV), generator=torch.Generator().manual_seed(1)).cpu()
        assert not torch.equal(other, got)


# ---------------------------------------------------------------------------------------------------
# StableDiffusionPipeline: a saved directory naming each scheduler loads and samples
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_pipeline_saved_with_sigma_scheduler_samples(tmp_path, kind, tiny):
    from b200sd import StableDiffusionPipeline
    from b200sd.pipeline import denoise_loop
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES
    cls = _classes(kind)[0]
    unet = UNet2DConditionModel(**TINY_OVERRIDES)
    unet.load_state_dict(tiny[1].state_dict(), strict=True)
    StableDiffusionPipeline(unet=unet, scheduler=cls(**_SD)).save_pretrained(str(tmp_path))
    pipe = StableDiffusionPipeline.from_pretrained(str(tmp_path)).to(DEV)
    assert type(pipe.scheduler) is cls
    ctx2 = torch.randn(4, 77, 64, generator=torch.Generator().manual_seed(4)).to(DEV)
    out = pipe(prompt_embeds=ctx2, height=256, width=256, num_inference_steps=8, guidance_scale=7.5,
               generator=torch.Generator(DEV).manual_seed(0), output_type="latent")
    assert pipe.unet._samplers, "the pipeline did not sample on the captured graph"
    g = torch.Generator(DEV).manual_seed(0)
    lat = torch.randn((2, 4, 32, 32), generator=g, device=DEV)
    want = denoise_loop(pipe.unet, cls(**_SD), lat, ctx2, 8, 7.5, record=[], generator=g)
    cos = _cos(out.images, want)
    assert out.images.shape == (2, 4, 32, 32) and torch.isfinite(out.images).all() and cos >= 0.9999, cos
