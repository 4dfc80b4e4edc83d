"""CPU tests of the host-side mirror of the diffusers surface: state-dict compatibility, scheduler
timestep tables and configuration behaviour, weight packing.  No GPU."""
import json
import os

import pytest
import torch

from oracle import schedulers_ref as R
from oracle import unet_ref as U


def test_facade_state_dict_is_diffusers_compatible():
    from b200sd.unet import UNet2DConditionModel
    ref = U.make_oracle_unet(seed=0, **U.TINY_OVERRIDES)
    m = UNet2DConditionModel(**U.TINY_OVERRIDES)
    sd, msd = ref.state_dict(), m.state_dict()
    assert list(sd.keys()) == list(msd.keys()) or set(sd) == set(msd)
    for k in sd:
        assert sd[k].shape == msd[k].shape, k
    m.load_state_dict(sd, strict=True)
    assert m.in_channels == 4 and m.config.cross_attention_dim == 64 and m.config["attention_head_dim"] == 2


def test_facade_full_size_key_set():
    from b200sd.unet import UNet2DConditionModel
    with torch.device("meta"):
        ref = U.UNet2DConditionModelRef()
    m = UNet2DConditionModel.__new__(UNet2DConditionModel)
    torch.nn.Module.__init__(m)
    # build on the meta device to avoid allocating 3.4 GB
    with torch.device("meta"):
        orig = UNet2DConditionModel.reset_parameters
        UNet2DConditionModel.reset_parameters = lambda self: None
        try:
            m = UNet2DConditionModel()
        finally:
            UNet2DConditionModel.reset_parameters = orig
    assert set(m.state_dict()) == set(ref.state_dict())
    assert sum(p.numel() for p in m.parameters()) == 859_520_964


def test_save_and_from_pretrained_roundtrip(tmp_path):
    from b200sd.unet import UNet2DConditionModel
    m = UNet2DConditionModel(**U.TINY_OVERRIDES)
    m.save_pretrained(str(tmp_path / "unet"))
    cfg = json.load(open(tmp_path / "unet" / "config.json"))
    assert cfg["_class_name"] == "UNet2DConditionModel" and cfg["cross_attention_dim"] == 64
    m2 = UNet2DConditionModel.from_pretrained(str(tmp_path), subfolder="unet")
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_unet_rejects_cpu_inputs_and_bad_config():
    from b200sd._lib import B200SDError
    from b200sd.unet import UNet2DConditionModel
    m = UNet2DConditionModel(**U.TINY_OVERRIDES).eval()
    with pytest.raises(B200SDError):
        m(torch.randn(1, 4, 16, 16), 1, torch.randn(1, 77, 64))      # CPU tensors: there is no CPU fallback
    with pytest.raises(TypeError):
        UNet2DConditionModel(not_a_field=1)
    with pytest.raises(NotImplementedError):
        UNet2DConditionModel(block_out_channels=(48, 96, 96, 96))


def test_scheduler_tables_match_oracle():
    from b200sd.schedulers import DDIMScheduler, DDPMScheduler, PNDMScheduler
    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    d = DDIMScheduler(clip_sample=False, set_alpha_to_one=False, **kw)
    r = R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False)
    assert torch.equal(d.alphas_cumprod, r.alphas_cumprod)
    for n in (50, 75, 20, 1000):
        d.set_timesteps(n)
        r.set_timesteps(n)
        assert d.timesteps.tolist() == r.timesteps.tolist()
    assert d.init_noise_sigma == 1.0 and d.num_train_timesteps == 1000 and d.config.num_train_timesteps == 1000
    x = torch.randn(2, 3)
    assert d.scale_model_input(x, 5) is x
    for off in (0, 1):
        p = PNDMScheduler(skip_prk_steps=True, steps_offset=off, **kw)
        rp = R.PNDMSchedulerRef(skip_prk_steps=True, steps_offset=off)
        p.set_timesteps(50)
        rp.set_timesteps(50)
        assert p.timesteps.tolist() == rp.timesteps.tolist() and len(p.timesteps) == 51
    assert DDPMScheduler(**kw).num_train_timesteps == 1000


def test_scheduler_config_errors_and_roundtrip(tmp_path):
    from b200sd.schedulers import DDIMScheduler, PNDMScheduler
    with pytest.raises(NotImplementedError):
        PNDMScheduler(skip_prk_steps=False)
    with pytest.raises(NotImplementedError):
        DDIMScheduler(clip_sample=True)
    with pytest.raises(TypeError):
        DDIMScheduler(bogus=1)
    d = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                      set_alpha_to_one=False)
    with pytest.raises(ValueError):
        d.step(torch.zeros(1), 10, torch.zeros(1))       # set_timesteps not called
    d.save_config(str(tmp_path / "scheduler"))
    d2 = DDIMScheduler.from_config(str(tmp_path), subfolder="scheduler")
    assert vars(d2.config) == vars(d.config)


def test_packing_layouts():
    from b200sd import packing
    w = torch.randn(6, 4, 3, 3)
    p = packing.pack_conv3x3(w).float()
    assert p.shape == (6, 36)
    assert torch.allclose(p[2, (1 * 3 + 2) * 4 + 3], w[2, 3, 1, 2].bfloat16().float())
    wg, bg = packing.pack_geglu(torch.arange(16.)[:, None].repeat(1, 2), torch.arange(16.), 8)
    # tile 8 -> [4 values | 4 gates] per tile: rows 0-3, 8-11, 4-7, 12-15
    assert bg.tolist() == [0, 1, 2, 3, 8, 9, 10, 11, 4, 5, 6, 7, 12, 13, 14, 15]
    assert wg[:, 0].float().tolist() == bg.tolist()


def test_fp32_path_weight_split_reconstructs_the_3_term_product():
    """engine_fp32._pack_lin / _pack_conv: [A_hi | A_lo] x [W_hi | W_hi]^T + A_hi x W_lo^T == A W^T to ~2^-16 (CPU, fp32 math)."""
    import torch
    from b200sd.engine_fp32 import _pack_conv, _pack_lin
    torch.manual_seed(0)
    A = torch.randn(64, 128)
    W = torch.randn(96, 128) / 11
    a_hi = A.bfloat16()
    a_lo = (A - a_hi.float()).bfloat16()
    w1, w2 = _pack_lin(W)
    assert w1.shape == (96, 256) and w2.shape == (96, 128) and w1.dtype == torch.bfloat16
    got = torch.cat([a_hi, a_lo], 1).float() @ w1.float().t() + a_hi.float() @ w2.float().t()
    want = A.double() @ W.double().t()
    rel = float((got.double() - want).abs().max() / want.abs().max())
    assert rel < 5e-5, rel
    plain = float(((a_hi.float() @ W.bfloat16().float().t()).double() - want).abs().max() / want.abs().max())
    assert plain > 20 * rel          # the single-term bf16 product is what the split improves on
    Wc = torch.randn(32, 64, 3, 3)
    c1, c2 = _pack_conv(Wc)
    assert c1.shape == (32, 18 * 64) and c2.shape == (32, 9 * 64)
    hi = Wc.permute(0, 2, 3, 1).reshape(32, 9, 64).bfloat16()
    assert torch.equal(c1.view(32, 9, 128)[:, :, :64], hi) and torch.equal(c1.view(32, 9, 128)[:, :, 64:], hi)
    assert torch.allclose(c1.view(32, 9, 128)[:, :, :64].float() + c2.view(32, 9, 64).float(), Wc.permute(0, 2, 3, 1).reshape(32, 9, 64),
                          rtol=0, atol=2e-4)


def test_fma_pipe_exp2_polynomial_model():
    """Numpy model of the attention kernel's FMA-pipe exponential (attention_tc.cu::poly_exp2x2): round-to-nearest split
    through the 1.5 * 2^23 magic constant, cubic on [-0.5, 0.5], exponent add on the bit pattern.  Pins the coefficients:
    relative error <= 1e-4 (P is rounded to bf16, 3.9e-3, right after) over the whole admissible range."""
    import numpy as np
    t = np.concatenate([np.linspace(-125.0, 6.0, 200001), np.array([-300.0, -125.0, -0.5, 0.0, 0.5, 6.0])]).astype(np.float32)
    tc = np.maximum(t, np.float32(-125.0))
    magic = np.float32(12582912.0)
    y = (tc + magic).astype(np.float32)
    ti = (y - magic).astype(np.float32)
    f = (tc - ti).astype(np.float32)
    assert np.all(np.abs(f) <= 0.5)
    c = [np.float32(v) for v in (0.9999280571937561, 0.6932609677314758, 0.2426111251115799, 0.0551716685295105)]
    q = (c[3] * f + c[2]).astype(np.float32)
    q = (q * f + c[1]).astype(np.float32)
    q = (q * f + c[0]).astype(np.float32)
    bits = ((y.view(np.uint32).astype(np.uint64) << np.uint64(23)) + q.view(np.uint32).astype(np.uint64)) & np.uint64(0xFFFFFFFF)
    e = bits.astype(np.uint32).view(np.float32)
    want = np.exp2(tc.astype(np.float64))
    rel = np.abs(e.astype(np.float64) - want) / want
    assert rel.max() <= 1e-4, rel.max()


def test_gn_parts_layouts_cover_every_sd_groupnorm():
    """ops.gn_parts_supported mirrors the G / Cg choice of b200sd_groupnorm_silu_parts: every GroupNorm width of the SD v1.5
    UNet (incl. the up-block concats) must be covered; a width the group count does not divide is refused."""
    import importlib
    ops = importlib.import_module("b200sd.ops")
    for C in (320, 640, 960, 1280, 1920, 2560):
        assert ops.gn_parts_supported(C, 32), C
    assert not ops.gn_parts_supported(330, 32)     # not divisible by the group count
    assert ops.gn_parts_supported(96, 32)          # 3 channels per group: 16 groups per CTA make 8-channel vectors


def test_bench_image_sharding():
    """bench.py --total-images: every image lands on exactly one rank, chunks differ by at most one, low ranks first."""
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for total in (1, 2, 3, 7, 8, 64):
        for world in (1, 2, 4, 8):
            parts = [bench.shard_images(total, world, r) for r in range(world)]
            assert sum(parts) == total and max(parts) - min(parts) <= 1
            assert parts == sorted(parts, reverse=True)


def test_bench_config_dicts_of_both_arms_are_one_function():
    """The driver compares the `config` of `bench.py` and `bench.py --impl reference` (same_config): both arms must build it from
    the same arguments with the same function, and it must name the workload without model-training keys."""
    import importlib.util, inspect, os
    spec = importlib.util.spec_from_file_location("bench_mod2", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    a = bench.sample_config(1, 1, 0, False)
    assert a["workload"] == "sd15_unet_ddim50_cfg7.5_512px" and a["unet_batch"] == 2 and a["total_images"] == 1
    assert bench.sample_config(1, 8, 0, False)["total_images"] == 8
    assert bench.sample_config(2, 4, 7, True)["workload"].endswith("512x768") and bench.sample_config(2, 4, 7, True)["total_images"] == 7
    src_ref, src_ours = inspect.getsource(bench.run_reference), inspect.getsource(bench.run_ours)
    assert '"config": sample_config(args.batch, args.gpus, args.total_images, args.portrait)' in src_ref
    assert '"config": sample_config(' in src_ours


def test_bench_dump_outputs_writes_float32_within_its_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files named after the outputs, whole when they fit; beyond DUMP_BYTES the same
    seeded sample of every output, so that two runs (two builds) stay comparable element for element."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod3", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    lat = torch.randn(2, 4, 8, 8, dtype=torch.float64)
    eps = torch.randn(4, 4, 8, 8, dtype=torch.bfloat16)
    bench.dump_outputs(str(tmp_path / "whole"), {"latents": lat, "noise_pred": eps})
    a, b = np.load(tmp_path / "whole" / "latents.npy"), np.load(tmp_path / "whole" / "noise_pred.npy")
    assert a.dtype == b.dtype == np.float32 and a.shape == (2, 4, 8, 8) and b.shape == (4, 4, 8, 8)
    assert np.array_equal(a, lat.float().numpy()) and np.array_equal(b, eps.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)           # the two outputs hold 6144 bytes
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"latents": lat, "noise_pred": eps})
    files = [tmp_path / d / f"{n}.npy" for d in ("s1", "s2") for n in ("latents", "noise_pred")]
    assert sum(os.path.getsize(f) for f in files[:2]) <= 4000
    s = [np.load(f) for f in files]
    assert np.array_equal(s[0], s[2]) and np.array_equal(s[1], s[3])
    assert s[0].dtype == s[1].dtype == np.float32 and 0 < s[0].size < lat.numel() and 0 < s[1].size < eps.numel()
    assert np.isin(s[0], lat.float().numpy()).all() and np.isin(s[1], eps.float().numpy()).all()


def test_pipeline_wrapper_save_load_layout(tmp_path):
    """finetune_sd.py:517-537 builds StableDiffusionPipeline(text_encoder=, vae=, unet=, tokenizer=, scheduler=, safety_checker=,
    feature_extractor=) and save_pretrained()s it; utils.py:187-191 loads it back with safety_checker=None: the diffusers directory
    layout (model_index.json + unet/ + scheduler/) round-trips, including the scheduler CLASS (B.6: a DDPMScheduler is what the
    training script saves)."""
    from b200sd import StableDiffusionPipeline
    from b200sd.schedulers import DDIMScheduler, DDPMScheduler, PNDMScheduler
    from b200sd.unet import UNet2DConditionModel
    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    unet = UNet2DConditionModel(**U.TINY_OVERRIDES)
    for sch in (DDPMScheduler(num_train_timesteps=1000, **kw), DDIMScheduler(clip_sample=False, set_alpha_to_one=False, **kw),
                PNDMScheduler(skip_prk_steps=True, **kw)):
        d = tmp_path / type(sch).__name__
        pipe = StableDiffusionPipeline(text_encoder=None, vae=None, unet=unet, tokenizer=None, scheduler=sch,
                                       safety_checker=None, feature_extractor=None)
        pipe.save_pretrained(str(d))
        index = json.load(open(d / "model_index.json"))
        assert index["_class_name"] == "StableDiffusionPipeline"
        assert index["unet"] == ["diffusers", "UNet2DConditionModel"] and index["scheduler"][1] == type(sch).__name__
        assert index["safety_checker"] == [None, None] and index["vae"] == [None, None]
        assert os.path.exists(d / "unet" / "config.json") and os.path.exists(d / "scheduler" / "scheduler_config.json")
        again = StableDiffusionPipeline.from_pretrained(str(d), safety_checker=None)
        assert type(again.scheduler) is type(sch)
        assert again.scheduler.config.beta_end == 0.012
        for (k, a), (_, b) in zip(unet.state_dict().items(), again.unet.state_dict().items()):
            assert torch.equal(a, b), k
        # inference.py:404-409: the scheduler can be overridden at load time
        swapped = StableDiffusionPipeline.from_pretrained(str(d), scheduler=DDIMScheduler(clip_sample=False, set_alpha_to_one=False, **kw))
        assert isinstance(swapped.scheduler, DDIMScheduler)
    with pytest.raises(ValueError):
        StableDiffusionPipeline(unet=None, scheduler=None)
    with pytest.raises(ValueError):       # diffusers' own message for sizes that are not multiples of 8
        pipe(prompt_embeds=torch.zeros(2, 77, 64), height=100, width=64)
    with pytest.raises(ValueError):       # strings need a tokenizer / text encoder
        pipe("a book cover")


def test_plms_plan_table_reproduces_the_oracle_pndm_scheduler():
    """PNDMScheduler.plms_plan(): the per-call rows that drive the captured PLMS kernel (weights, eps-ring slots, saved-sample
    flags, cx / ce), executed here in plain torch on a random eps sequence, must walk the same trajectory as the oracle's
    PNDMScheduler (skip_prk_steps=True) -- including the repeated first timestep and the 4-deep history."""
    import torch
    from b200sd.schedulers import PNDMScheduler
    from oracle import schedulers_ref as R
    for steps, offset in ((50, 1), (50, 0), (7, 1), (4, 0)):
        ours = PNDMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", skip_prk_steps=True, steps_offset=offset)
        ours.set_timesteps(steps)
        ref = R.PNDMSchedulerRef(skip_prk_steps=True, steps_offset=offset)
        ref.set_timesteps(steps)
        assert ours.timesteps.tolist() == ref.timesteps.tolist() and len(ours.timesteps) == steps + 1
        rows = ours.plms_plan()
        assert len(rows) == steps + 1 and all(len(r) == 12 for r in rows)
        g = torch.Generator().manual_seed(steps)
        x = torch.randn(2, 4, 4, 4, generator=g, dtype=torch.float64)
        want = x.clone()
        ring, saved = [None] * 4, None
        for k, t in enumerate(ref.timesteps):
            eps = torch.randn(2, 4, 4, 4, generator=g, dtype=torch.float64)
            want = ref.step(eps, t, want).prev_sample
            w, (cx, ce), h, (slot, from_saved, save_x) = rows[k][:4], rows[k][4:6], [int(v) for v in rows[k][6:9]], rows[k][9:]
            acc = w[0] * eps + sum(w[1 + i] * ring[h[i]] for i in range(3) if h[i] >= 0)
            xv = saved if from_saved else x
            if save_x:
                saved = x.clone()
            x = cx * xv - ce * acc
            if slot >= 0:
                assert int(slot) not in [v for v in h if v >= 0]      # this call's eps never overwrites a slot it reads
                ring[int(slot)] = eps
            assert float((x - want).abs().max()) <= 2e-6 * max(1.0, float(want.abs().max())), (steps, offset, k)   # the oracle keeps its alpha table in fp32


def test_bench_reference_arm_prints_exactly_one_json_line_on_stdout():
    """The driver contract: stdout carries ONE JSON line.  The reference arm (the fp32 oracle on the host cores) runs here without
    a GPU; anything else the process writes to file descriptor 1 (C-level writers such as NCCL's banner at N > 1) is moved onto
    stderr by bench._claim_stdout()."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import os, sys; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0']; "
            "import bench; bench._claim_stdout(); os.write(1, b'NCCL version 0.0 (noise written to fd 1 by a C library)\\n'); bench.main()")
    r = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "unet_denoise_it_per_s" and d["unit"] == "it/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    assert d["config"]["workload"] == "sd15_unet_ddim50_cfg7.5_512px" and d["config"]["unet_batch"] == 2
    assert "NCCL version 0.0" in r.stderr
