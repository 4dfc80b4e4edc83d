"""Host side of ancestral sampling (DDPMScheduler; DDIMScheduler with eta > 0): timesteps, per-step coefficient rows and noise
rows against the fp32 oracle restatement of diffusers 0.7.2, the noise-draw contract, the DDPM == DDIM(eta = 1) equivalence,
and reloading a pipeline saved with a DDPMScheduler.  CPU only."""
import numpy as np
import pytest
import torch

from oracle import ancestral_ref as A

_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")


def _ddpm(**kw):
    from b200sd.schedulers import DDPMScheduler
    return DDPMScheduler(num_train_timesteps=1000, **_KW, **kw)


def _close(got, want, rel=1e-6):
    assert abs(got - want) <= rel * max(abs(want), 1e-30), (got, want)


@pytest.mark.parametrize("n", [1, 7, 20, 50, 1000, 1200])
def test_ddpm_timesteps_match_oracle(n):
    ours, ref = _ddpm(), A.DDPMSchedulerRef()
    ours.set_timesteps(n)
    ref.set_timesteps(n)
    assert ours.timesteps.dtype == torch.int64
    assert ours.timesteps.tolist() == ref.timesteps.tolist()
    assert ours.num_inference_steps == ref.num_inference_steps == min(1000, n)


@pytest.mark.parametrize("n", [50, 1000])
@pytest.mark.parametrize("variance_type", ["fixed_small", "fixed_large"])
@pytest.mark.parametrize("clip", [True, False])
def test_ddpm_rows_match_oracle(n, variance_type, clip):
    ours, ref = _ddpm(variance_type=variance_type, clip_sample=clip), A.DDPMSchedulerRef(variance_type=variance_type,
                                                                                         clip_sample=clip)
    ours.set_timesteps(n)
    ref.set_timesteps(n)
    rows, n_noisy = ours.ancestral_plan()
    assert len(rows) == len(ref.timesteps) and n_noisy == sum(1 for t in ref.timesteps.tolist() if t > 0)
    k = 0
    for row, t in zip(rows, ref.timesteps.tolist()):
        row = torch.tensor(row, dtype=torch.float32).tolist()          # what the device table holds
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noise_row, clip_flag = row
        a_t = ref.alphas_cumprod[t]
        _close(sa_t, float(a_t ** 0.5))
        _close(sb_t, float((1 - a_t) ** 0.5))
        want_x0, want_x = ref.coefficients(t)
        _close(c_x0, float(want_x0))
        _close(c_x, float(want_x))
        assert c_e == 0.0
        if t > 0:
            _close(c_z, float(ref._get_variance(t) ** 0.5))
            assert noise_row == k
            k += 1
        else:
            assert noise_row == -1.0 and c_z == 0.0
        assert clip_flag == float(clip)


@pytest.mark.parametrize("eta", [0.5, 1.0])
@pytest.mark.parametrize("set_alpha_to_one", [True, False])
def test_ddim_eta_rows_match_oracle(eta, set_alpha_to_one):
    from b200sd.schedulers import DDIMScheduler
    ours = DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=set_alpha_to_one)
    ref = A.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=set_alpha_to_one)
    ours.set_timesteps(50)
    ref.set_timesteps(50)
    # the oracle's formulas on its fp32 abar table, evaluated in fp64 like the facade: in fp32, sqrt(1 - a_p - sigma^2)
    # cancels to ~1e-5 relative error at eta = 1
    ref.alphas_cumprod = ref.alphas_cumprod.double()
    ref.final_alpha_cumprod = ref.final_alpha_cumprod.double()
    rows, n_noisy = ours.ancestral_plan(eta)
    assert n_noisy == len(rows) == 50
    ratio = 1000 // 50
    for k, (row, t) in enumerate(zip(rows, ref.timesteps.tolist())):
        row = torch.tensor(row, dtype=torch.float32).tolist()
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noise_row, clip_flag = row
        prev_t = t - ratio
        a_t = ref.alphas_cumprod[t]
        a_p = ref.alphas_cumprod[prev_t] if prev_t >= 0 else ref.final_alpha_cumprod
        std = eta * ref._get_variance(t, prev_t) ** 0.5
        _close(sa_t, float(a_t ** 0.5))
        _close(sb_t, float((1 - a_t) ** 0.5))
        _close(c_x0, float(a_p ** 0.5))
        assert c_x == 0.0
        _close(c_e, float((1 - a_p - std ** 2) ** 0.5))
        if float(std) == 0.0:
            assert c_z == 0.0
        else:
            _close(c_z, float(std))
        assert noise_row == k and clip_flag == 0.0


@pytest.mark.parametrize("n", [50, 1000])
@pytest.mark.parametrize("set_alpha_to_one", [True, False])
def test_ddim_eta0_rows_are_the_deterministic_ddim_update(n, set_alpha_to_one):
    """At eta = 0 the affine row is DDIM's update, sqrt(a_p) x0 + sqrt(1 - a_p) eps, with no x term, no noise and no clipping:
    sa_t, sb_t, c_x0, c_e equal sa_t, sb_t, sa_p, sb_p of DDIM's closed form below (what b200sd_cfg_ddim_step takes), exactly
    in fp64 and after rounding to the fp32 the kernel receives."""
    from b200sd.schedulers import DDIMScheduler
    ours = DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=set_alpha_to_one)
    ours.set_timesteps(n)

    def ddim_coefs(t):
        prev_t = t - ours.num_train_timesteps // ours.num_inference_steps
        a_t, a_p = ours._ac[t], ours._ac[prev_t] if prev_t >= 0 else ours._final_alpha
        return a_t ** 0.5, (1 - a_t) ** 0.5, a_p ** 0.5, (1 - a_p) ** 0.5

    rows, n_noisy = ours.ancestral_plan(0.0)
    assert n_noisy == 0 and len(rows) == n
    for row, t in zip(rows, ours.timesteps.tolist()):
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noisy, clip = ours._ancestral_coefs(t, 0.0)
        assert c_x == 0.0 and c_z == 0.0 and not noisy and not clip
        want = ddim_coefs(t)
        assert (sa_t, sb_t, c_x0, c_e) == want
        f32 = lambda v: torch.tensor(v, dtype=torch.float32).tolist()
        assert f32([sa_t, sb_t, c_x0, c_e]) == f32(list(want))
        assert f32(row) == f32([*want[:3], 0.0, want[3], 0.0, -1.0, 0.0])


def test_ddim_eta_out_of_range_raises():
    from b200sd.schedulers import DDIMScheduler
    s = DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=False)
    s.set_timesteps(50)
    with pytest.raises(ValueError):
        s.ancestral_plan(1.5)


def test_step_noise_matches_oracle_draws():
    from b200sd.schedulers import step_noise
    sample = torch.zeros(2, 4, 8, 8)
    g_ours, g_ref = torch.Generator().manual_seed(5), torch.Generator().manual_seed(5)
    for _ in range(4):
        assert torch.equal(step_noise(sample, g_ours), A.step_noise(sample, g_ref))
    torch.manual_seed(6)
    a = step_noise(sample)
    torch.manual_seed(6)
    assert torch.equal(a, A.step_noise(sample))
    assert a.dtype == torch.float32 and a.shape == sample.shape


def test_ddpm_equals_ddim_eta1_at_1000_steps_in_the_oracle():
    """DDPM ancestral sampling (fixed_small, no clipping) is DDIM with eta = 1 at every training timestep: the two
    restatements agree step for step on the same noise.  The beta / abar tables are rebuilt in fp64 so that this checks the
    algebra.  On the fp32 tables the identity a_t / a_p = alpha_t only holds to the cumprod's rounding, which is ~1e-4 of
    beta_t near t = 0, and the two fp32 loops end 3e-5 (max-abs over max-abs) apart."""
    ddpm = A.DDPMSchedulerRef(variance_type="fixed_small", clip_sample=False)
    ddim = A.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=True)
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float64) ** 2
    for s in (ddpm, ddim):
        s.betas, s.alphas, s.alphas_cumprod = betas, 1.0 - betas, torch.cumprod(1.0 - betas, dim=0)
    ddpm.one, ddim.final_alpha_cumprod = ddpm.one.double(), ddim.final_alpha_cumprod.double()
    ddpm.set_timesteps(1000)
    ddim.set_timesteps(1000)
    assert ddpm.timesteps.tolist() == ddim.timesteps.tolist()
    x0 = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(0)).double()
    eps_model = lambda x, t: 0.8 * torch.tanh(x) + 0.1 * np.sin(t / 50.0)
    ga, gb = torch.Generator().manual_seed(1), torch.Generator().manual_seed(1)
    xa, xb = x0.clone(), x0.clone()
    for t in ddpm.timesteps.tolist():
        xa = ddpm.step(eps_model(xa, t), t, xa, generator=ga).prev_sample
        xb = ddim.step(eps_model(xb, t), t, xb, eta=1.0, generator=gb).prev_sample
        torch.testing.assert_close(xa, xb, rtol=1e-5, atol=1e-5 * float(xb.abs().max()))


def test_unsupported_variance_types_raise():
    for vt in ("learned", "learned_range", "fixed_small_log"):
        s = _ddpm(variance_type=vt)          # still constructs: add_noise does not need it
        with pytest.raises(NotImplementedError):
            s.set_timesteps(50)


def test_pipeline_saved_with_ddpm_reloads_with_a_sampling_scheduler(tmp_path):
    from b200sd.pipeline import StableDiffusionPipeline
    from b200sd.schedulers import DDPMScheduler
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES
    pipe = StableDiffusionPipeline(unet=UNet2DConditionModel(**TINY_OVERRIDES), scheduler=_ddpm())
    pipe.save_pretrained(str(tmp_path))
    again = StableDiffusionPipeline.from_pretrained(str(tmp_path))
    assert isinstance(again.scheduler, DDPMScheduler)
    again.scheduler.set_timesteps(50)
    assert again.scheduler.timesteps.tolist() == list(range(980, -1, -20))
    rows, n_noisy = again.scheduler.ancestral_plan()
    assert len(rows) == 50 and n_noisy == 49
