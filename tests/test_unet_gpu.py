"""GPU parity of the whole UNet forward and of the 50-step CFG sampling loop against the fp32 oracle
on identical random-init weights (seed 0; default torch init, to_q/to_k x4 -- oracle.unet_ref
make_oracle_unet: default torch init, to_q/to_k x2), latents, timesteps and context.

Tolerances (BASELINE.json north_star): bf16 noise prediction max|x-ref|/max|ref| <= 1e-2;
50-step sampled latents cosine >= 0.999."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rel(got, want):
    return float((got.float().cpu() - want.float().cpu()).abs().max() / want.float().abs().max())


@pytest.fixture(scope="module")
def models():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    oracle = make_oracle_unet(seed=0)
    ours = UNet2DConditionModel()
    ours.load_state_dict(oracle.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    return oracle, ours


def test_config1_single_forward_vs_cpu_oracle(models):
    """BASELINE config 1: batch 1, 4x64x64 latent, 77x768 context, oracle fp32 on CPU."""
    oracle, ours = models
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 64, 64, generator=g)
    ctx = torch.randn(1, 77, 768, generator=g)
    for t in (1, 500, 981):
        with torch.no_grad():
            want = oracle(x, t, ctx).sample
            got = ours(x.to(DEV), t, ctx.to(DEV)).sample
        assert got.shape == want.shape and got.dtype == torch.float32
        r = _rel(got, want)
        assert r <= 1e-2, f"t={t}: max-rel {r:.4g}"


def test_batch2_per_sample_timesteps_and_graph_equivalence(models):
    oracle, ours = models
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 4, 64, 64, generator=g)
    ctx = torch.randn(2, 77, 768, generator=g)
    t = torch.tensor([980, 20])
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = oc(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample
            ours.use_cuda_graph = False
            eager = ours(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample
            ours.use_cuda_graph = True
            g1 = ours(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample
            g2 = ours(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample
    finally:
        oracle.to("cpu")
        ours.use_cuda_graph = True
    assert _rel(eager, want) <= 1e-2
    # every kernel (incl. split-K and GroupNorm reductions) sums in a fixed order: bit-reproducible
    assert torch.equal(eager, g1) and torch.equal(g1, g2), "graph replay must be bit-identical to eager launches"


def test_portrait_latent_96x64(models):
    """BASELINE config 5 geometry (512 wide x 768 high -> 4x96x64 latent)."""
    oracle, ours = models
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 4, 96, 64, generator=g)
    ctx = torch.randn(2, 77, 768, generator=g)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = oc(x.to(DEV), 500, ctx.to(DEV)).sample
            got = ours(x.to(DEV), 500, ctx.to(DEV)).sample
    finally:
        oracle.to("cpu")
    assert _rel(got, want) <= 1e-2


def test_50_step_cfg_ddim_sampling_cosine(models):
    """BASELINE config 2: 50-step DDIM, CFG 7.5, batch-1 image (UNet batch 2).  The oracle loop runs in
    fp32 on the GPU (same oracle module, moved to CUDA with TF32 off) so the test finishes in seconds."""
    from b200sd.pipeline import denoise_loop
    from b200sd.schedulers import DDIMScheduler
    from oracle import schedulers_ref as R
    oracle, ours = models
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            rec_ref, rec = [], []
            ref_s = R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False)
            want = R.denoise_loop(oc, ref_s, lat.to(DEV), ctx2.to(DEV), 50, 7.5, record=rec_ref)
            sch = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                                set_alpha_to_one=False)
            got = denoise_loop(ours, sch, lat.to(DEV), ctx2.to(DEV), 50, 7.5, record=rec)
    finally:
        oracle.to("cpu")
    cos = float(torch.nn.functional.cosine_similarity(got.flatten().float(), want.flatten().float(), dim=0))
    assert cos >= 0.999, f"50-step latents cosine {cos:.6f}"
    # note: the CFG-combined eps (recorded per step) amplifies the difference eps_c - eps_u by 7.5x, so its
    # max-rel error is ~7.5*sqrt(2) times the UNet's; the UNet output itself is bounded by the tests above.


def test_per_step_unet_eps_along_the_50_step_trajectory(models):
    """BASELINE config 2 / SURVEY 8(d): "each-step eps vs oracle (bf16 1e-2)".  Along OUR 50-step CFG-7.5 DDIM trajectory, the
    UNet output of every step (the raw (2, 4, 64, 64) noise prediction, BEFORE the CFG combine) is compared with the fp32 oracle
    evaluated on the SAME input latents / timestep / context: per-step max-rel <= 1e-2 at all 50 steps."""
    from b200sd.schedulers import DDIMScheduler
    oracle, ours = models
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(1, 4, 64, 64, generator=g).to(DEV)
    ctx2 = torch.randn(2, 77, 768, generator=g).to(DEV)
    sch = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, set_alpha_to_one=False)
    sch.set_timesteps(50)
    oc = oracle.to(DEV)
    worst = (0.0, None)
    try:
        with torch.no_grad():
            for t in sch.timesteps.tolist():
                x2 = torch.cat([lat, lat])
                eps2 = ours(x2, t, ctx2).sample
                want = oc(x2, t, ctx2).sample
                r = _rel(eps2, want)
                worst = max(worst, (r, t))
                assert r <= 1e-2, f"step t={t}: UNet eps max-rel {r:.4g}"
                lat = sch.step_cfg(eps2, t, lat, 7.5).prev_sample
    finally:
        oracle.to("cpu")
    print(f"per-step UNet eps along the trajectory: worst max-rel {worst[0]:.4g} at t={worst[1]}")


def test_config1_margin_over_five_input_seeds(models):
    """The bf16 bar (1e-2 max-rel) on five more (latent, context, timestep) draws, reported with the maximum: the margin of the
    full-size random-init network is thin (0.85-1.0e-2 in round 1), so one lucky seed is not evidence."""
    oracle, ours = models
    oc = oracle.to(DEV)
    rels = []
    try:
        with torch.no_grad():
            for seed in range(10, 15):
                g = torch.Generator().manual_seed(seed)
                x = torch.randn(2, 4, 64, 64, generator=g).to(DEV)
                ctx = torch.randn(2, 77, 768, generator=g).to(DEV)
                t = torch.randint(0, 1000, (2,), generator=g).to(DEV)
                rels.append(_rel(ours(x, t, ctx).sample, oc(x, t, ctx).sample))
    finally:
        oracle.to("cpu")
    print("config-1 bf16 max-rel over 5 seeds:", [f"{r:.4g}" for r in rels], "max", f"{max(rels):.4g}")
    assert max(rels) <= 1e-2, rels


def test_large_batch_plan_batch8(models):
    """UNet batch >= 8 switches two ends of the plan to the tensor cores (all 22 time_emb_proj heads as one GEMM; conv_out as an
    implicit GEMM with hi | lo split weights) and every GEMM grid becomes multi-round (persistent kernel): same 1e-2 bar."""
    oracle, ours = models
    g = torch.Generator().manual_seed(21)
    x = torch.randn(8, 4, 64, 64, generator=g).to(DEV)
    ctx = torch.randn(8, 77, 768, generator=g).to(DEV)
    t = torch.randint(0, 1000, (8,), generator=g).to(DEV)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = oc(x, t, ctx).sample
            got = ours(x, t, ctx).sample
    finally:
        oracle.to("cpu")
    r = _rel(got, want)
    print(f"batch-8 plan max-rel {r:.4g}")
    assert r <= 1e-2, r


def test_50_step_cfg_plms_sampling_cosine(models):
    from b200sd.pipeline import denoise_loop
    from b200sd.schedulers import PNDMScheduler
    from oracle import schedulers_ref as R
    oracle, ours = models
    g = torch.Generator().manual_seed(43)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = R.denoise_loop(oc, R.PNDMSchedulerRef(skip_prk_steps=True, steps_offset=1), lat.to(DEV), ctx2.to(DEV), 50, 7.5)
            sch = PNDMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", skip_prk_steps=True,
                                steps_offset=1)
            got = denoise_loop(ours, sch, lat.to(DEV), ctx2.to(DEV), 50, 7.5)
    finally:
        oracle.to("cpu")
    cos = float(torch.nn.functional.cosine_similarity(got.flatten().float(), want.flatten().float(), dim=0))
    assert cos >= 0.999, f"51-call PLMS latents cosine {cos:.6f}"


def test_sharp_attention_stress_not_worse_than_library_bf16():
    """Stress recipe (to_q/to_k x4): the random network amplifies bf16 operand rounding far beyond 1e-2
    for ANY bf16 implementation.  Requirement here: our error <= the torch eager bf16 (cuDNN/cuBLAS)
    error of the same oracle module, both measured against the fp32 oracle."""
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet
    oracle = make_oracle_unet(seed=0, sharpen_attention=4.0)
    ours = UNet2DConditionModel()
    ours.load_state_dict(oracle.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    oracle = oracle.to(DEV)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 4, 64, 64, generator=g).to(DEV)
    ctx = torch.randn(2, 77, 768, generator=g).to(DEV)
    with torch.no_grad():
        want = oracle(x, 500, ctx).sample
        got = ours(x, 500, ctx).sample
        lib_bf16 = oracle.bfloat16()(x.bfloat16(), 500, ctx.bfloat16()).sample.float()
    e_ours, e_lib = _rel(got, want), _rel(lib_bf16, want)
    assert e_ours <= e_lib and e_ours < 0.1, f"ours {e_ours:.4g} vs torch-bf16 {e_lib:.4g}"


def test_forward_rejects_bad_inputs(models):
    _, ours = models
    with pytest.raises(ValueError):
        ours(torch.randn(1, 3, 64, 64, device=DEV), 1, torch.randn(1, 77, 768, device=DEV))
    with pytest.raises(ValueError):
        ours(torch.randn(1, 4, 60, 64, device=DEV), 1, torch.randn(1, 77, 768, device=DEV))
    with pytest.raises(ValueError):
        ours(torch.randn(2, 4, 64, 64, device=DEV), 1, torch.randn(1, 77, 768, device=DEV))


def test_fp32_accuracy_path_within_1e_4(models):
    """BASELINE north_star: "the fp32 path within 1e-4".  unet.set_precision("fp32") evaluates every contraction as a 3-term
    split-bf16 product with fp32 accumulation on the same tcgen05 kernels (engine_fp32.py)."""
    oracle, ours = models
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 4, 64, 64, generator=g)
    ctx = torch.randn(2, 77, 768, generator=g)
    t = torch.tensor([999, 37])
    oc = oracle.to(DEV)
    ours.set_precision("fp32")
    try:
        with torch.no_grad():
            want = oc(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample
            got = ours(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample
            again = ours(x.to(DEV), t.to(DEV), ctx.to(DEV)).sample      # graph replay
    finally:
        oracle.to("cpu")
        ours.set_precision("bf16")
    r = _rel(got, want)
    print(f"fp32 path max-rel vs fp32 oracle: {r:.3g}")
    assert r <= 1e-4, f"fp32 path max-rel {r:.4g}"
    assert torch.equal(got, again)


def test_context_cache_is_not_fooled_by_address_reuse(models):
    """The engine projects the context to K/V once per context tensor.  A NEW context that the caching allocator places at
    the freed address of the previous one (same shape, version 0) must not be taken for the old one."""
    _, ours = models
    g = torch.Generator().manual_seed(7)
    x = torch.randn(2, 4, 64, 64, generator=g).to(DEV)
    ctx_a = torch.randn(2, 77, 768, generator=g).to(DEV)
    ctx_b_host = torch.randn(2, 77, 768, generator=g)
    with torch.no_grad():
        ours(x, 500, ctx_a)
        ptr_a = ctx_a.data_ptr()
        del ctx_a
        ctx_b = ctx_b_host.to(DEV)                    # usually lands on ctx_a's block
        got = ours(x, 500, ctx_b).sample.clone()
        same_address = ctx_b.data_ptr() == ptr_a
        want = ours(x, 500, ctx_b.clone()).sample     # a different object: always re-projected
    assert torch.equal(got, want), f"stale context K/V (address reused: {same_address})"


# ---------------------------------------------------------------------------------------------------
# CapturedSampler: the whole denoising step as one CUDA graph
# ---------------------------------------------------------------------------------------------------
_DDIM_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, set_alpha_to_one=False)


@pytest.fixture(scope="module")
def oracle_50_step(models):
    from oracle import schedulers_ref as R
    oracle, _ours = models
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = R.denoise_loop(oc, R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), lat.to(DEV), ctx2.to(DEV), 50, 7.5)
    finally:
        oracle.to("cpu")
    return lat, ctx2, want.cpu()


def test_captured_sampler_50_steps_vs_oracle(models, oracle_50_step):
    """BASELINE config 2 through the one-graph-per-step sampler (what bench.py times): 50-step latents cosine >= 0.999 vs the
    fp32 oracle loop."""
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    _oracle, ours = models
    lat, ctx2, want = oracle_50_step
    sch = DDIMScheduler(**_DDIM_KW)
    sch.set_timesteps(50)
    smp = CapturedSampler(ours, sch, 1, 64, 64, 77, 7.5, lanes=1)
    got = smp.run(lat.to(DEV), ctx2.to(DEV)).cpu()
    cos = float(torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0))
    assert cos >= 0.999, f"50-step latents cosine {cos:.6f}"
    # the same sampler object again, other latents first: no state leaks between runs (cursor, context K/V, latents)
    smp.run(torch.randn(1, 4, 64, 64).to(DEV), ctx2.flip(0).to(DEV))
    again = smp.run(lat.to(DEV), ctx2.to(DEV)).cpu()
    assert torch.equal(again, got), "a second run of the captured sampler on the same inputs must be bit-identical"


def test_denoise_loop_takes_the_captured_sampler_and_matches_the_per_call_loop(models, oracle_50_step):
    from b200sd.pipeline import denoise_loop
    from b200sd.schedulers import DDIMScheduler
    _oracle, ours = models
    lat, ctx2, want = oracle_50_step
    rec = []
    per_call = denoise_loop(ours, DDIMScheduler(**_DDIM_KW), lat.to(DEV), ctx2.to(DEV), 50, 7.5, record=rec).cpu()   # record -> per-call loop
    captured = denoise_loop(ours, DDIMScheduler(**_DDIM_KW), lat.to(DEV), ctx2.to(DEV), 50, 7.5).cpu()
    assert getattr(ours, "_samplers", None), "denoise_loop did not build a CapturedSampler"
    cos = float(torch.nn.functional.cosine_similarity(captured.flatten(), per_call.flatten(), dim=0))
    assert cos >= 0.9995, f"captured vs per-call loop cosine {cos:.6f}"
    cos_o = float(torch.nn.functional.cosine_similarity(captured.flatten(), want.flatten(), dim=0))
    assert cos_o >= 0.999


def test_captured_sampler_host_step_equals_device_steps(models):
    """host_step(): H2D latents + context out of pinned buffers, context K/V, step, D2H -- the same numbers as step()."""
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    _oracle, ours = models
    g = torch.Generator().manual_seed(7)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    sch = DDIMScheduler(**_DDIM_KW)
    sch.set_timesteps(50)
    smp = CapturedSampler(ours, sch, 1, 64, 64, 77, 7.5)
    smp.set_context(ctx2.to(DEV))
    smp.set_latents(lat.to(DEV))
    smp.reset(0)
    for _ in range(3):
        smp.step()
    want = smp.latents.cpu()
    lat_h, ctx_h, out_h = lat.clone().pin_memory(), ctx2.clone().pin_memory(), torch.empty(1, 4, 64, 64).pin_memory()
    smp.bind_host(lat_h, ctx_h, out_h)
    smp.reset(0)
    for _ in range(3):
        smp.host_step()
        lat_h.copy_(out_h)
    assert torch.equal(out_h, want)


def test_captured_sampler_refuses_stale_weights(models):
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    from b200sd._lib import B200SDError
    _oracle, ours = models
    sch = DDIMScheduler(**_DDIM_KW)
    sch.set_timesteps(4)
    smp = CapturedSampler(ours, sch, 1, 64, 64, 77, 7.5)
    w = ours.conv_out.bias
    with torch.no_grad():
        w.add_(1.0)
    try:
        with pytest.raises(B200SDError):
            smp.run(torch.randn(1, 4, 64, 64).to(DEV), torch.randn(2, 77, 768).to(DEV))
    finally:
        with torch.no_grad():
            w.sub_(1.0)


def test_captured_sampler_batched_portrait_tiny_net():
    """2 images (UNet batch 4) at a portrait geometry on the reduced-width network reproduce the oracle loop."""
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    from b200sd.unet import UNet2DConditionModel
    from oracle import schedulers_ref as R
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    oracle = make_oracle_unet(seed=0, **TINY_OVERRIDES)
    ours = UNet2DConditionModel(**TINY_OVERRIDES)
    ours.load_state_dict(oracle.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(2, 4, 48, 32, generator=g)
    ctx2 = torch.randn(4, 77, 64, generator=g)
    with torch.no_grad():
        want = R.denoise_loop(oracle, R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False), lat, ctx2, 6, 7.5)
    sch = DDIMScheduler(**_DDIM_KW)
    sch.set_timesteps(6)
    got = CapturedSampler(ours, sch, 2, 48, 32, 77, 7.5, lanes=1).run(lat.to(DEV), ctx2.to(DEV)).cpu()
    cos = float(torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0))
    assert cos >= 0.999, f"cosine {cos:.6f}"
    with pytest.raises(ValueError, match="lanes=2"):
        CapturedSampler(ours, sch, 2, 48, 32, 77, 7.5, lanes=2)


def test_captured_sampler_plms_51_calls_vs_oracle_and_per_call_loop(models):
    """utils.py:222-224: PNDM skip_prk_steps=True (PLMS).  The captured sampler replays all 51 UNet calls (the first timestep
    twice) as the same CUDA graph with the eps history in a device ring: latents cosine >= 0.999 vs the fp32 oracle loop and
    ~equal to our per-call loop."""
    from b200sd.pipeline import denoise_loop
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import PNDMScheduler
    from oracle import schedulers_ref as R
    oracle, ours = models
    g = torch.Generator().manual_seed(11)
    lat = torch.randn(1, 4, 64, 64, generator=g)
    ctx2 = torch.randn(2, 77, 768, generator=g)
    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", skip_prk_steps=True, steps_offset=1)
    oc = oracle.to(DEV)
    try:
        with torch.no_grad():
            want = R.denoise_loop(oc, R.PNDMSchedulerRef(skip_prk_steps=True, steps_offset=1), lat.to(DEV), ctx2.to(DEV), 50, 7.5).cpu()
    finally:
        oracle.to("cpu")
    sch = PNDMScheduler(**kw)
    sch.set_timesteps(50)
    smp = CapturedSampler(ours, sch, 1, 64, 64, 77, 7.5)
    assert smp.n_steps == 51
    got = smp.run(lat.to(DEV), ctx2.to(DEV)).cpu()
    cos = float(torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0))
    assert cos >= 0.999, f"captured PLMS latents cosine {cos:.6f}"
    assert torch.equal(smp.run(lat.to(DEV), ctx2.to(DEV)).cpu(), got)          # ring / saved sample / cursor fully re-armed
    rec = []
    per_call = denoise_loop(ours, PNDMScheduler(**kw), lat.to(DEV), ctx2.to(DEV), 50, 7.5, record=rec).cpu()
    cos2 = float(torch.nn.functional.cosine_similarity(got.flatten(), per_call.flatten(), dim=0))
    assert cos2 >= 0.9999, f"captured vs per-call PLMS cosine {cos2:.6f}"
    via_loop = denoise_loop(ours, PNDMScheduler(**kw), lat.to(DEV), ctx2.to(DEV), 50, 7.5).cpu()     # takes the captured sampler
    assert torch.equal(via_loop, got)
