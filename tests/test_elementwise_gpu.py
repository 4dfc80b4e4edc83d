"""GPU parity of the scheduler / loss elementwise kernels against the oracle (fp32: 1e-6 relative,
bf16 storage: 1 bf16 ulp of the result)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import schedulers_ref as R


def _dev():
    return torch.device("cuda:0")


@pytest.mark.parametrize("n_shape", [(1, 4, 64, 64), (3, 4, 96, 64), (1, 4, 5, 7), (2, 3, 1, 1)])
@pytest.mark.parametrize("cfg", [True, False])
def test_cfg_ddim_step_fp32(n_shape, cfg):
    from b200sd import ops
    torch.manual_seed(0)
    B = n_shape[0]
    x = torch.randn(n_shape)
    eps2 = torch.randn((2 * B if cfg else B,) + n_shape[1:])
    sch = R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False)
    sch.set_timesteps(50)
    for t in (980, 500, 0):
        eps = R.cfg_combine(eps2, 7.5) if cfg else eps2
        want = sch.step(eps, t, x).prev_sample
        a_t = float(sch.alphas_cumprod[t])
        p = t - 20
        a_p = float(sch.alphas_cumprod[p]) if p >= 0 else float(sch.final_alpha_cumprod)
        e2 = eps2.to(_dev())
        eu, ec = (e2[:B].contiguous(), e2[B:].contiguous()) if cfg else (e2, None)
        got = ops.cfg_ddim_step(eu, ec, x.to(_dev()), 7.5, a_t ** 0.5, (1 - a_t) ** 0.5, a_p ** 0.5, (1 - a_p) ** 0.5)
        torch.testing.assert_close(got.cpu(), want, rtol=2e-6, atol=2e-6 * float(want.abs().max()))


def test_cfg_ddim_step_bf16_eps():
    from b200sd import ops
    torch.manual_seed(1)
    x = torch.randn(2, 4, 64, 64)
    e2 = torch.randn(4, 4, 64, 64).bfloat16()
    sch = R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False)
    sch.set_timesteps(50)
    t = 500
    want = sch.step(R.cfg_combine(e2.float(), 7.5), t, x).prev_sample
    a_t, a_p = float(sch.alphas_cumprod[t]), float(sch.alphas_cumprod[t - 20])
    d = e2.to(_dev())
    got = ops.cfg_ddim_step(d[:2].contiguous(), d[2:].contiguous(), x.to(_dev()), 7.5, a_t ** 0.5, (1 - a_t) ** 0.5,
                            a_p ** 0.5, (1 - a_p) ** 0.5)
    torch.testing.assert_close(got.cpu(), want, rtol=2e-6, atol=1e-5)


@pytest.mark.parametrize("steps_offset", [0, 1])
def test_plms_loop_matches_oracle(steps_offset):
    """Full 51-call PLMS trajectory with a fake eps model: facade scheduler vs oracle scheduler."""
    from b200sd.schedulers import PNDMScheduler
    torch.manual_seed(2)
    x = torch.randn(2, 4, 16, 16)
    ref = R.PNDMSchedulerRef(skip_prk_steps=True, steps_offset=steps_offset)
    ours = PNDMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", skip_prk_steps=True,
                         steps_offset=steps_offset)
    ref.set_timesteps(50)
    ours.set_timesteps(50)
    assert ours.timesteps.tolist() == ref.timesteps.tolist()
    xr, xo = x.clone(), x.to(_dev())
    for i, t in enumerate(ref.timesteps):
        g = torch.Generator().manual_seed(100 + i)
        eps = torch.randn(x.shape, generator=g)
        xr = ref.step(eps, t, xr).prev_sample
        xo = ours.step(eps.to(_dev()), t, xo).prev_sample
        torch.testing.assert_close(xo.cpu(), xr, rtol=1e-5, atol=1e-5 * float(xr.abs().max()))


def test_ddim_facade_loop_matches_oracle():
    from b200sd.schedulers import DDIMScheduler
    torch.manual_seed(3)
    x = torch.randn(1, 4, 64, 64)
    ref = R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False)
    ours = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                         set_alpha_to_one=False)
    ref.set_timesteps(50)
    ours.set_timesteps(50)
    assert ours.timesteps.tolist() == ref.timesteps.tolist()
    xr, xo = x.clone(), x.to(_dev())
    for i, t in enumerate(ref.timesteps):
        eps = torch.randn(x.shape, generator=torch.Generator().manual_seed(i))
        xr = ref.step(eps, t, xr).prev_sample
        xo = ours.step(eps.to(_dev()), t, xo).prev_sample
    torch.testing.assert_close(xo.cpu(), xr, rtol=1e-5, atol=1e-5 * float(xr.abs().max()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_add_noise(dtype):
    from b200sd.schedulers import DDPMScheduler
    torch.manual_seed(4)
    x0 = torch.randn(8, 4, 64, 64).to(dtype)
    noise = torch.randn(8, 4, 64, 64).to(dtype)
    t = torch.tensor([0, 1, 20, 500, 980, 981, 999, 333])
    ref = R.DDPMSchedulerRef()
    ours = DDPMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    want = ref.add_noise(x0.float(), noise.float(), t)
    got = ours.add_noise(x0.to(_dev()), noise.to(_dev()), t.to(_dev()))
    assert got.dtype == dtype
    tol = 1e-6 if dtype == torch.float32 else 8e-3
    torch.testing.assert_close(got.float().cpu(), want, rtol=tol, atol=tol)


@pytest.mark.parametrize("shape", [(8, 4, 64, 64), (1, 4, 3, 5), (2, 4, 96, 64)])
def test_mse_loss_fwd_bwd(shape):
    from b200sd import ops
    torch.manual_seed(5)
    pred = torch.randn(shape, requires_grad=True)
    tgt = torch.randn(shape)
    want = R.mse_loss_ref(pred, tgt)
    want.backward()
    p = pred.detach().to(_dev()).requires_grad_(True)
    got = ops.mse_loss(p, tgt.to(_dev()))
    got.backward()
    torch.testing.assert_close(got.detach().cpu(), want.detach(), rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(p.grad.cpu(), pred.grad, rtol=1e-5, atol=1e-9)
    # repeat: the self-cleaning workspace counter must allow back-to-back launches
    got2 = ops.mse_loss(p.detach(), tgt.to(_dev()))
    torch.testing.assert_close(got2.cpu(), want.detach(), rtol=1e-5, atol=1e-7)


def test_bad_inputs_raise():
    from b200sd import ops
    from b200sd._lib import B200SDError
    x = torch.randn(4, 4)
    with pytest.raises(B200SDError):
        ops.cfg_ddim_step(x, None, x, 7.5, 1.0, 0.0, 1.0, 0.0)  # CPU tensors: no fallback
    xd = x.to(_dev())
    with pytest.raises(ValueError):
        ops.cfg_ddim_step(xd, None, torch.randn(5, 4, device=_dev()), 7.5, 1.0, 0.0, 1.0, 0.0)


# ---- the CUDA scheduler kernels against diffusers 0.7.2's OWN known answers (tests/golden/diffusers_0_7_2_kat.json;
# ---- recipes in tests/test_oracle_diffusers_kat.py): not oracle-vs-kernel but published-vector-vs-kernel


@pytest.mark.parametrize("variant", ["no_noise", "set_alpha_to_one", "no_set_alpha_to_one"])
def test_ddim_kernel_reproduces_diffusers_full_loop_known_answer(variant):
    from b200sd.schedulers import DDIMScheduler
    from test_oracle_diffusers_kat import SCHED_CFG, VARIANTS, _check_sched, dummy_model, dummy_sample_deter
    # clip_sample=False (the reference's setting, inference.py:386-387): the clamp of diffusers' test config never binds here
    sch = DDIMScheduler(**{**SCHED_CFG, "clip_sample": False, **VARIANTS[variant]})
    sch.set_timesteps(10)
    sample = dummy_sample_deter().contiguous().to(_dev())
    for t in sch.timesteps:
        sample = sch.step(dummy_model(sample, t).contiguous(), t, sample, eta=0.0).prev_sample
    assert isinstance(sch.step(sample, 0, sample, return_dict=False), tuple)
    _check_sched("ddim", variant, sample.cpu())


@pytest.mark.parametrize("variant", ["no_noise", "set_alpha_to_one", "no_set_alpha_to_one"])
def test_plms_kernel_reproduces_diffusers_full_loop_known_answer(variant):
    """diffusers' test enters PLMS through 12 Runge-Kutta calls, which the reference skips (utils.py:222-224) and the product
    refuses; they run on the oracle, the 7 `step_plms` calls (4th-order branch, `_get_prev_sample`) run on the CUDA kernel."""
    from b200sd.schedulers import PNDMScheduler
    from test_oracle_diffusers_kat import SCHED_CFG, VARIANTS, _check_sched, dummy_model, dummy_sample_deter
    cfg = {**SCHED_CFG, "skip_prk_steps": True, **VARIANTS[variant]}
    warm = R.PNDMSchedulerRef(**cfg)
    warm.set_timesteps(10)
    sample, plms_timesteps = R.pndm_prk_warmup(warm, dummy_model, dummy_sample_deter())
    sch = PNDMScheduler(**cfg)
    sch.set_timesteps(10)
    sch.ets, sch.counter = [e.contiguous().to(_dev()) for e in warm.ets], warm.counter
    sample = sample.contiguous().to(_dev())
    for t in plms_timesteps:
        sample = sch.step(dummy_model(sample, int(t)).contiguous(), int(t), sample, return_dict=False)[0]   # diffusers' tuple form
    _check_sched("pndm", variant, sample.cpu())
