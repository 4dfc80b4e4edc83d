"""Host side of the image-to-image and legacy inpainting pipelines: where a run enters the schedule for a given strength, the
sliced coefficient plans of the captured sampler, PIL preprocessing, argument validation and loading a saved
StableDiffusionPipeline into both classes.  Against the fp32 restatement of diffusers 0.7.2 in oracle/img2img_ref.py.  CPU only."""
import numpy as np
import pytest
import torch

from oracle import ancestral_ref as A
from oracle import img2img_ref as I
from oracle import schedulers_ref as R

_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
_KINDS = ["ddim_offset0", "ddim_offset1", "plms_offset1", "ddpm"]


def _pair(kind):
    """(ours, oracle) schedulers of one kind, set_timesteps not yet called"""
    from b200sd.schedulers import DDIMScheduler, DDPMScheduler, PNDMScheduler
    if kind.startswith("ddim"):
        off = int(kind[-1])
        return (DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=False, steps_offset=off),
                R.DDIMSchedulerRef(clip_sample=False, set_alpha_to_one=False, steps_offset=off))
    if kind == "plms_offset1":
        return (PNDMScheduler(**_KW, skip_prk_steps=True, steps_offset=1),
                R.PNDMSchedulerRef(skip_prk_steps=True, steps_offset=1))
    return DDPMScheduler(num_train_timesteps=1000, **_KW), A.DDPMSchedulerRef()


@pytest.mark.parametrize("strength", [0.0, 0.29, 0.75, 1.0])
@pytest.mark.parametrize("n", [1, 10, 50])
@pytest.mark.parametrize("kind", _KINDS)
def test_start_and_sliced_timesteps_match_oracle(kind, n, strength):
    ours, ref = _pair(kind)
    t_start, t_noise = ours.img2img_start(n, strength)
    r_start, r_noise = I.img2img_start(ref, n, strength)
    assert (t_start, t_noise) == (r_start, r_noise)
    assert ours.timesteps[t_start:].tolist() == ref.timesteps[r_start:].tolist()
    offset = 1 if kind.endswith("1") else 0
    init_timestep = min(int(n * strength) + offset, n)
    assert t_start == max(n - init_timestep + offset, 0)
    assert t_noise == int(ours.timesteps[-init_timestep])


def test_start_keeps_the_0_7_2_arithmetic():
    """int(50 * 0.29) is 14 in Python floats; init_timestep 0 noises to timesteps[0]"""
    ours, _ = _pair("ddim_offset0")
    assert ours.img2img_start(50, 0.29) == (36, int(ours.timesteps[-14]))
    assert ours.img2img_start(50, 0.0) == (50, int(ours.timesteps[0]))
    assert ours.img2img_start(50, 1.0) == (0, int(ours.timesteps[-50]))


@pytest.mark.parametrize("strength", [-0.01, 1.01])
def test_strength_out_of_range_raises(strength):
    ours, _ = _pair("ddim_offset0")
    with pytest.raises(ValueError):
        ours.img2img_start(50, strength)


def _old_ancestral_plan(s, eta):
    """ancestral_plan before `start` existed"""
    rows, k = [], 0
    for t in s.timesteps.tolist():
        sa_t, sb_t, c_x0, c_x, c_e, c_z, noisy, clip = s._ancestral_coefs(t, eta)
        rows.append([sa_t, sb_t, c_x0, c_x, c_e, c_z, float(k if noisy else -1), float(clip)])
        k += noisy
    return rows, k


@pytest.mark.parametrize("kind,eta", [("ddpm", 0.0), ("ddim_offset0", 0.0), ("ddim_offset0", 1.0), ("ddim_offset1", 0.5)])
@pytest.mark.parametrize("start", [0, 1, 13, 49, 50])
def test_ancestral_plan_start_is_the_slice_with_renumbered_noise_rows(kind, eta, start):
    ours, _ = _pair(kind)
    ours.set_timesteps(50)
    full, n_full = ours.ancestral_plan(eta)
    assert (full, n_full) == _old_ancestral_plan(ours, eta)
    rows, n_noisy = ours.ancestral_plan(eta, start)
    assert len(rows) == 50 - start
    k = 0
    for row, want in zip(rows, full[start:]):
        assert row[:6] == want[:6] and row[7] == want[7]
        if want[6] < 0:
            assert row[6] == -1.0
        else:
            assert row[6] == k
            k += 1
    assert n_noisy == k


def _old_plms_plan(s):
    """plms_plan before `start` existed"""
    rows, ets = [], []
    for counter, timestep in enumerate(s.timesteps.tolist()):
        ets, keep_eps, w, hist, cx, ce, save_x, from_saved = s._plms_call(counter, timestep, ets)
        slot = -1
        if keep_eps:
            slot = next(k for k in range(4) if k not in ets)
            ets.append(slot)
        rows.append(w + [0.0] * (4 - len(w)) + [cx, ce] + [float(h) for h in hist] + [-1.0] * (3 - len(hist))
                    + [float(slot), float(from_saved), float(save_x)])
    return rows


def _run_plms_rows(rows, dim):
    """What cfg_plms_step_table computes, row by row, on symbolic vectors: the sample is basis vector 0, the eps of call k is
    basis vector k + 1.  Returns the sample after every call."""
    x, saved, ring, out = np.eye(dim)[0], np.zeros(dim), np.zeros((4, dim)), []
    for k, row in enumerate(rows):
        w, cx, ce = row[:4], row[4], row[5]
        hist, slot, from_saved, save_x = [int(h) for h in row[6:9]], int(row[9]), row[10] != 0, row[11] != 0
        e = np.eye(dim)[k + 1]
        acc = w[0] * e
        for j, h in enumerate(hist):
            if h >= 0:
                acc = acc + w[1 + j] * ring[h]
        xv = saved if from_saved else x
        if save_x:
            saved = x.copy()
        x = cx * xv - ce * acc
        if slot >= 0:
            ring[slot] = e
        out.append(x)
    return out


@pytest.mark.parametrize("n,strength", [(50, 0.75), (50, 0.29), (10, 1.0), (10, 0.1), (3, 0.75), (1, 1.0)])
def test_plms_plan_start_matches_the_oracle_stepped_over_the_slice(n, strength):
    ours, ref = _pair("plms_offset1")
    t_start, _ = ours.img2img_start(n, strength)
    assert ours.plms_plan() == _old_plms_plan(ours)
    rows = ours.plms_plan(t_start)
    I.img2img_start(ref, n, strength)
    ts = ref.timesteps.tolist()
    assert len(rows) == len(ts) - t_start
    # the counter rule applied to the slice, call by call
    ets = []
    for counter, (row, t) in enumerate(zip(rows, ts[t_start:])):
        ets, keep_eps, w, hist, cx, ce, save_x, from_saved = ours._plms_call(counter, t, ets)
        assert row[:4] == w + [0.0] * (4 - len(w)) and row[4:6] == [cx, ce]
        assert row[10:] == [float(from_saved), float(save_x)]
        ets = ets + ([len(ets)] if keep_eps else [])
    # the oracle's PNDM step, counter starting at 0 on timesteps[t_start], on the same symbolic vectors
    dim = len(rows) + 1
    got = _run_plms_rows(rows, dim)
    x = torch.eye(dim, dtype=torch.float64)[0]
    for k, t in enumerate(ref.timesteps[t_start:]):
        x = ref.step(torch.eye(dim, dtype=torch.float64)[k + 1], t, x).prev_sample
        np.testing.assert_allclose(got[k], x.numpy(), rtol=2e-6, atol=2e-6 * float(x.abs().max()))


def _rgb(w, h, seed=0):
    from PIL import Image
    return Image.fromarray(np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8), "RGB")


@pytest.mark.parametrize("w,h", [(64, 64), (100, 77), (513, 250), (256, 384)])
def test_pil_preprocessing_matches_numpy_restatement(w, h):
    from PIL import Image
    from b200sd.pipeline import preprocess_image, preprocess_mask
    img = preprocess_image(_rgb(w, h))
    assert img.dtype == torch.float32 and tuple(img.shape) == (1, 3, h - h % 32, w - w % 32)
    assert torch.equal(img, I.preprocess_image(_rgb(w, h)))
    assert float(img.min()) >= -1.0 and float(img.max()) <= 1.0
    gray = Image.fromarray(np.random.default_rng(1).integers(0, 256, (h, w), dtype=np.uint8), "L")
    for m in (gray, gray.convert("RGB")):
        mask = preprocess_mask(m)
        assert tuple(mask.shape) == (1, 4, (h - h % 32) // 8, (w - w % 32) // 8)
        assert torch.equal(mask, I.preprocess_mask(m))
    white = preprocess_mask(Image.new("L", (w, h), 255))
    black = preprocess_mask(Image.new("L", (w, h), 0))
    assert torch.equal(white, torch.zeros_like(white)) and torch.equal(black, torch.ones_like(black))   # white = repaint


def _cpu_pipe(cls):
    from b200sd.schedulers import DDIMScheduler
    from b200sd.unet import UNet2DConditionModel
    from b200sd.vae import AutoencoderKL
    from oracle.unet_ref import TINY_OVERRIDES
    from oracle.vae_ref import TINY_VAE_OVERRIDES
    return cls(vae=AutoencoderKL(**TINY_VAE_OVERRIDES), unet=UNet2DConditionModel(**TINY_OVERRIDES),
               scheduler=DDIMScheduler(**_KW, clip_sample=False, set_alpha_to_one=False))


def test_argument_validation():
    from PIL import Image
    from b200sd import StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy
    img2img, inpaint = _cpu_pipe(StableDiffusionImg2ImgPipeline), _cpu_pipe(StableDiffusionInpaintPipelineLegacy)
    ctx2 = torch.zeros(4, 77, 64)                 # two prompts
    img = torch.zeros(1, 3, 256, 256)
    for s in (-0.5, 1.5):
        with pytest.raises(ValueError, match="strength"):
            img2img(prompt_embeds=ctx2, init_image=img, strength=s)
        with pytest.raises(ValueError, match="strength"):
            inpaint(prompt_embeds=ctx2, init_image=img, mask_image=torch.ones(1, 4, 32, 32), strength=s)
    with pytest.raises(ValueError, match="batch"):
        img2img(prompt_embeds=ctx2, init_image=torch.zeros(3, 3, 256, 256))
    with pytest.raises(ValueError, match="multiples of 8"):
        img2img(prompt_embeds=ctx2, init_image=torch.zeros(1, 3, 252, 256))
    with pytest.raises(ValueError, match="same size"):
        inpaint(prompt_embeds=ctx2, init_image=img, mask_image=torch.ones(1, 4, 16, 32))
    with pytest.raises(ValueError, match="same size"):
        inpaint(prompt_embeds=ctx2, init_image=img, mask_image=torch.ones(3, 4, 32, 32))
    with pytest.raises(ValueError, match="same size"):
        inpaint(prompt_embeds=ctx2, init_image=_rgb(256, 256), mask_image=Image.new("L", (256, 320), 255))
    with pytest.raises(ValueError, match="mask_image"):
        inpaint(prompt_embeds=ctx2, init_image=img)
    with pytest.raises(TypeError):
        img2img(prompt_embeds=ctx2, init_image=img, height=512)
    with pytest.raises(TypeError):
        inpaint(prompt_embeds=ctx2, init_image=img, mask_image=torch.ones(1, 4, 32, 32), num_images_per_prompt=2)


def test_saved_text_to_image_pipeline_loads_into_both_classes(tmp_path):
    from b200sd import StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy, StableDiffusionPipeline
    from b200sd.schedulers import DDIMScheduler
    from b200sd.vae import AutoencoderKL
    _cpu_pipe(StableDiffusionPipeline).save_pretrained(str(tmp_path))
    for cls in (StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy):
        pipe = cls.from_pretrained(str(tmp_path))
        assert type(pipe) is cls and isinstance(pipe, StableDiffusionPipeline)
        assert isinstance(pipe.scheduler, DDIMScheduler) and isinstance(pipe.vae, AutoencoderKL)
