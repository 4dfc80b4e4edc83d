"""Host side of the sigma-space schedulers (LMSDiscreteScheduler, EulerDiscreteScheduler, EulerAncestralDiscreteScheduler), no
GPU: the timestep and sigma tables against diffusers 0.7.2's construction (oracle/sigma_ref.py), the captured sampler's plan
against the per-call step rule, the LMS coefficients against the oracle's, two float64 identities that tie Euler and
Euler-ancestral to DDIM (eta = 0 and eta = 1) independently of any recalled number, the published known answers reproduced by
the oracle, and what is refused."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import sigma_ref as S

HERE = os.path.dirname(os.path.abspath(__file__))
KAT = json.load(open(os.path.join(HERE, "golden", "diffusers_0_7_2_sigma_kat.json")))
_SD = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
_KAT_CFG = dict(num_train_timesteps=1100, beta_start=0.0001, beta_end=0.02, beta_schedule="linear")
KINDS = ("lms", "euler", "euler_ancestral")


def _classes(kind):
    from b200sd import schedulers as B
    return {"lms": (B.LMSDiscreteScheduler, S.LMSDiscreteSchedulerRef),
            "euler": (B.EulerDiscreteScheduler, S.EulerDiscreteSchedulerRef),
            "euler_ancestral": (B.EulerAncestralDiscreteScheduler, S.EulerAncestralDiscreteSchedulerRef)}[kind]


def _pair(kind, n, **cfg):
    ours_cls, ref_cls = _classes(kind)
    ours, ref = ours_cls(**cfg), ref_cls(**cfg)
    ours.set_timesteps(n)
    ref.set_timesteps(n)
    return ours, ref


# ---------------------------------------------------------------------------------------------------
# tables
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("cfg", [_SD, _KAT_CFG, {}])
@pytest.mark.parametrize("n", [1, 10, 25, 50, 1000])
def test_timestep_and_sigma_tables_match_0_7_2(kind, cfg, n):
    ours, ref = _pair(kind, n, **cfg)
    assert ours.timesteps.dtype == torch.float64 and torch.equal(ours.timesteps, ref.timesteps)
    assert ours.sigmas.dtype == torch.float32 and torch.equal(ours.sigmas, ref.sigmas)
    assert ours.init_noise_sigma == float(ref.init_noise_sigma)
    assert len(ours.sigmas) == n + 1 and float(ours.sigmas[-1]) == 0.0


def test_tables_before_set_timesteps_match_0_7_2():
    for kind in KINDS:
        ours_cls, ref_cls = _classes(kind)
        ours, ref = ours_cls(**_SD), ref_cls(**_SD)
        assert torch.equal(ours.timesteps, ref.timesteps) and torch.equal(ours.sigmas, ref.sigmas)


@pytest.mark.parametrize("kind", KINDS)
def test_scale_model_input_equals_oracle_bit_for_bit(kind):
    ours, ref = _pair(kind, 50, **_SD)
    x = torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(0))
    for t in ref.timesteps:
        assert torch.equal(ours.scale_model_input(x, t), ref.scale_model_input(x, t))
        assert torch.equal(ours.scale_model_input(x, float(t)), ref.scale_model_input(x, t))


def test_unknown_timestep_raises():
    ours, _ = _pair("euler", 50, **_SD)
    t = float(ours.timesteps[1])
    assert t != int(t)
    with pytest.raises(ValueError):
        ours.scale_model_input(torch.zeros(1), int(t))
    with pytest.raises(ValueError):
        ours.scale_model_input(torch.zeros(1), torch.tensor(t, dtype=torch.float32))     # rounded to fp32: not in the table


# ---------------------------------------------------------------------------------------------------
# the step rule: the captured sampler's plan is the per-call rule, step by step
# ---------------------------------------------------------------------------------------------------
def _diffusers_history(n, order):
    """0.7.2 LMS's derivative list, with each derivative named by its step index: per step, the entries the update reads
    (newest first, this step's first)"""
    derivs, reads = [], []
    for i in range(n):
        derivs.append(i)
        if len(derivs) > order:
            derivs.pop(0)
        o = min(i + 1, order)
        reads.append(list(reversed(derivs))[:o])
    return reads


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [10, 25, 50, 1000])
@pytest.mark.parametrize("order", [1, 2, 3, 4])
def test_sigma_plan_rows_are_the_per_call_rule(kind, n, order):
    ours, _ = _pair(kind, n, **_SD)
    rows, n_noise = ours.sigma_plan(order)
    assert len(rows) == n and all(len(r) == 12 for r in rows)
    reads = _diffusers_history(n, order)
    hist, ring, k = [], {}, 0          # the per-call step: history entries are the step index of the derivative
    for i, row in enumerate(rows):
        hist, sigma, coefs, used, keep, noisy, sigma_up = ours._sigma_call(i, hist, order)
        assert row[0] == np.float32(sigma) and row[0] == float(ours.sigmas[i])
        assert row[1:1 + len(coefs)] == [float(c) for c in coefs] and all(c == 0.0 for c in row[1 + len(coefs):5])
        slots = [int(s) for s in row[5:8]]
        assert [s for s in slots if s >= 0] == slots[:len(used)] and all(s < 0 for s in slots[len(used):])
        assert [ring[s] for s in slots[:len(used)]] == used            # the ring slots hold the derivatives the rule reads
        if kind == "lms":
            assert [i] + used == reads[i]                               # ... which are the ones 0.7.2 reads
            assert len(coefs) == min(i + 1, order)
        else:
            assert used == [] and len(coefs) == 1
        slot = int(row[8])
        assert (slot >= 0) == keep == (kind == "lms" and order > 1)
        if keep:
            assert slot not in [s for s, step in ring.items() if step in hist]   # never overwrites a live entry
            ring[slot] = i
            hist.append(i)
        assert int(row[9]) == (k if noisy else -1) and noisy == (kind == "euler_ancestral")
        assert row[10] == float(sigma_up) and row[11] == float(ours._in_div[i])
        k += noisy
    assert n_noise == k == (n if kind == "euler_ancestral" else 0)


@pytest.mark.parametrize("n", [10, 25])
def test_lms_coefficients_equal_the_oracle(n):
    ours, ref = _pair("lms", n, **_SD)
    for i in range(n):
        o = min(i + 1, 4)
        got, _, _ = ours._coefs(i, 4, ours._sig)
        want = [ref.get_lms_coefficient(o, i, k) for k in range(o)]
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)


def test_in_div_is_torchs_fp32_formula():
    ours, ref = _pair("euler_ancestral", 50, **_SD)
    for i, t in enumerate(ref.timesteps):
        sigma = ref.sigmas[i]
        assert float(ours._in_div[i]) == float((sigma ** 2 + 1) ** 0.5)


def test_euler_ancestral_sigma_up_down_are_torchs_fp32():
    ours, ref = _pair("euler_ancestral", 50, **_SD)
    for i in range(50):
        coefs, noisy, sigma_up = ours._coefs(i, 4, ours._sig)
        sf, st = ref.sigmas[i], ref.sigmas[i + 1]
        up = (st ** 2 * (sf ** 2 - st ** 2) / sf ** 2) ** 0.5
        down = (st ** 2 - up ** 2) ** 0.5
        assert float(sigma_up) == float(up) and float(coefs[0]) == float(down - sf) and noisy
    assert float(ours._coefs(49, 4, ours._sig)[2]) == 0.0


# ---------------------------------------------------------------------------------------------------
# float64 identities: one step in VE variables at DDIM's integer timesteps equals DDIM's step
# ---------------------------------------------------------------------------------------------------
def _ddim_and_sigmas(n=50):
    from b200sd.schedulers import DDIMScheduler
    ddim = DDIMScheduler(**_SD, clip_sample=False, set_alpha_to_one=True)
    ddim.set_timesteps(n)
    ts = ddim.timesteps.tolist()
    abar = [ddim._ac[t] for t in ts] + [1.0]            # set_alpha_to_one: abar_prev of the last step is 1
    sig = np.array([((1 - a) / a) ** 0.5 for a in abar], dtype=np.float64)
    return ddim, ts, abar, sig


def _ve_step(x, e, sigma, coefs, sigma_up, z):
    x0 = x - sigma * e
    d = (x - x0) / sigma
    return x + coefs[0] * d + sigma_up * z


@pytest.mark.parametrize("kind,eta", [("euler", 0.0), ("euler_ancestral", 1.0)])
def test_fp64_step_equals_ddim(kind, eta):
    ddim, ts, abar, sig = _ddim_and_sigmas()
    sch = _classes(kind)[0](**_SD)
    g = torch.Generator().manual_seed(0)
    for i, t in enumerate(ts):
        x_vp = torch.randn(64, generator=g, dtype=torch.float64)
        e = torch.randn(64, generator=g, dtype=torch.float64)
        z = torch.randn(64, generator=g, dtype=torch.float64)
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noisy, clip = ddim._ancestral_coefs(t, eta)
        want = c_x0 * (x_vp - sb_t * e) / sa_t + c_x * x_vp + c_e * e + (c_z * z if noisy else 0)
        _, sigma, coefs, _, _, noisy_ve, sigma_up = sch._sigma_call(i, [], 1, sig=sig)
        assert noisy_ve == (eta > 0)
        got = _ve_step(x_vp / abar[i] ** 0.5, e, sigma, coefs, sigma_up, z) * abar[i + 1] ** 0.5
        torch.testing.assert_close(got, want, rtol=1e-12, atol=1e-12 * float(want.abs().max()))


def test_lms_order_1_is_euler():
    from b200sd.schedulers import EulerDiscreteScheduler, LMSDiscreteScheduler
    _, _, _, sig = _ddim_and_sigmas()
    lms, euler = LMSDiscreteScheduler(**_SD), EulerDiscreteScheduler(**_SD)
    for i in range(50):
        c_lms = lms._sigma_call(i, [], 1, sig=sig)[2]
        c_eul = euler._sigma_call(i, [], 1, sig=sig)[2]
        np.testing.assert_allclose(c_lms, c_eul, rtol=1e-12)
    lms.set_timesteps(50)
    euler.set_timesteps(50)
    rl, re = lms.sigma_plan(1)[0], euler.sigma_plan(1)[0]
    for a, b in zip(rl, re):
        np.testing.assert_allclose(a[1], b[1], rtol=1e-6)       # quad's integral of 1 vs the fp32 difference
        assert a[:1] + a[2:] == b[:1] + b[2:]


# ---------------------------------------------------------------------------------------------------
# the published answers of diffusers 0.7.2's test suite, reproduced by the oracle
# ---------------------------------------------------------------------------------------------------
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


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_reproduces_published_full_loop(kind):
    ref = _classes(kind)[1](**_KAT_CFG)
    kw = {"generator": torch.manual_seed(0)} if kind == "euler_ancestral" else {}
    sample = kat_full_loop(ref, kw)
    want_sum, want_mean = KAT[kind]
    assert abs(float(sample.abs().sum()) - want_sum) < KAT["tolerances"]["sum_atol"]
    assert abs(float(sample.abs().mean()) - want_mean) < KAT["tolerances"]["mean_atol"]


# ---------------------------------------------------------------------------------------------------
# configuration and what is refused
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_config_round_trip(kind, tmp_path):
    cls = _classes(kind)[0]
    cls(**_SD).save_config(str(tmp_path))
    cfg = json.load(open(tmp_path / "scheduler_config.json"))
    assert cfg["_class_name"] == cls.__name__
    again = cls.from_config(str(tmp_path))
    again.set_timesteps(30)
    ours, _ = _pair(kind, 30, **_SD)
    assert torch.equal(again.sigmas, ours.sigmas)


@pytest.mark.parametrize("kind", KINDS)
def test_refusals(kind):
    from b200sd.pipeline import StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy
    from b200sd.sampler import CapturedSampler
    ours, _ = _pair(kind, 10, **_SD)
    with pytest.raises(NotImplementedError):
        ours.add_noise(torch.zeros(1, 4), torch.zeros(1, 4), torch.tensor([5]))
    with pytest.raises(NotImplementedError):
        ours.img2img_start(10, 0.5)
    image, ctx2 = torch.zeros(1, 3, 64, 64), torch.zeros(2, 77, 8)
    with pytest.raises(NotImplementedError):
        StableDiffusionImg2ImgPipeline(unet=object(), scheduler=ours)(prompt_embeds=ctx2, init_image=image)
    with pytest.raises(NotImplementedError):
        StableDiffusionInpaintPipelineLegacy(unet=object(), scheduler=ours)(prompt_embeds=ctx2, init_image=image,
                                                                            mask_image=torch.ones(1, 4, 8, 8))
    with pytest.raises(ValueError):
        CapturedSampler(object(), ours, 1, 8, 8, start=1)
    with pytest.raises(ValueError):
        CapturedSampler(object(), ours, 1, 8, 8, inpaint=True)
    with pytest.raises(ValueError):
        ours._sigma_call(0, [], 5)


def test_euler_churn_is_refused():
    ours, _ = _pair("euler", 10, **_SD)
    t = ours.timesteps[0]
    with pytest.raises(NotImplementedError):
        ours.step(torch.zeros(4), t, torch.zeros(4), s_churn=1.0)
    ours._check_churn(t, 1.0, 0.0, 0.5)      # sigma outside [s_tmin, s_tmax]: gamma = 0, the plain Euler step


def test_pipeline_loader_admits_the_sigma_schedulers():
    from b200sd import EulerAncestralDiscreteScheduler, EulerDiscreteScheduler, LMSDiscreteScheduler
    from b200sd.pipeline import _SCHEDULERS
    for cls in (LMSDiscreteScheduler, EulerDiscreteScheduler, EulerAncestralDiscreteScheduler):
        assert cls.__name__ in _SCHEDULERS
