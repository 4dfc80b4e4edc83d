"""Host side of the 9-channel inpainting UNet and StableDiffusionInpaintPipeline: mask and masked-image preparation and the
latent-size mask against the fp32 restatement of diffusers 0.7.2 (oracle/inpaint_ref.py), the UNet's parameter set, argument
validation of the pipelines and of the captured sampler, and a saved directory loading into the new class.  CPU only."""
import json

import numpy as np
import pytest
import torch

from oracle import inpaint_ref as P9

_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")


def _pil_pair(w, h, seed=0):
    """an RGB picture and an "L" mask holding every grey level, 127 and 128 (either side of the 0.5 threshold) included"""
    from PIL import Image
    rng = np.random.default_rng(seed)
    image = Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), "RGB")
    grey = (np.arange(h * w) % 256).astype(np.uint8).reshape(h, w)
    grey[0, :2] = (127, 128)
    return image, Image.fromarray(grey, "L")


@pytest.mark.parametrize("w,h", [(64, 64), (96, 40), (24, 72)])
def test_prepare_mask_and_masked_image_matches_oracle(w, h):
    from b200sd.pipeline import prepare_mask_and_masked_image
    image, mask = _pil_pair(w, h, seed=w + h)
    m, mi = prepare_mask_and_masked_image(image, mask)
    rm, rmi = P9.prepare_mask_and_masked_image(image, mask)
    assert m.dtype == mi.dtype == torch.float32
    assert tuple(m.shape) == (1, 1, h, w) and tuple(mi.shape) == (1, 3, h, w)
    assert torch.equal(m, rm) and torch.equal(mi, rmi)
    assert float(m[0, 0, 0, 0]) == 0.0 and float(m[0, 0, 0, 1]) == 1.0        # grey 127 keeps, grey 128 repaints
    assert set(m.unique().tolist()) == {0.0, 1.0}
    assert float(mi.min()) >= -1.0 and float(mi.max()) <= 1.0


def test_prepare_tensor_inputs_binarise_like_pil():
    from b200sd.pipeline import prepare_mask_and_masked_image
    image, mask = _pil_pair(40, 24, seed=3)
    rm, rmi = P9.prepare_mask_and_masked_image(image, mask)
    img_t = torch.from_numpy(np.array(image)[None].transpose(0, 3, 1, 2).copy()).float() / 127.5 - 1.0
    mask_t = torch.from_numpy(np.array(mask)[None, None].copy()).float() / 255.0
    m, mi = prepare_mask_and_masked_image(img_t, mask_t)
    assert torch.equal(m, rm) and torch.equal(mi, rmi)
    # a batch of masks against one image broadcasts to the mask batch
    m2, mi2 = prepare_mask_and_masked_image(img_t, torch.cat([mask_t, 1 - mask_t]))
    assert tuple(mi2.shape) == (2, 3, 24, 40) and torch.equal(mi2[:1], rmi)


@pytest.mark.parametrize("H,W", [(512, 512), (768, 512), (200, 328)])
def test_latent_mask_is_torch_nearest_like_the_oracle(H, W):
    from b200sd.pipeline import latent_mask
    _, mask = _pil_pair(W, H, seed=H)
    m, _ = P9.prepare_mask_and_masked_image(_pil_pair(W, H)[0], mask)
    got, want = latent_mask(m, H // 8, W // 8), P9.latent_mask(m, H // 8, W // 8)
    assert tuple(got.shape) == (1, 1, H // 8, W // 8) and torch.equal(got, want)
    # nearest: every latent pixel is the top-left pixel of its 8 x 8 block
    assert torch.equal(got, m[:, :, ::8, ::8])


def test_nine_channel_unet_parameters():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import UNet2DConditionModelRef
    with torch.device("meta"):
        m = UNet2DConditionModel(in_channels=9)
        ref = UNet2DConditionModelRef(in_channels=9)
    sd, rsd = m.state_dict(), ref.state_dict()
    assert len(sd) == 686 and set(sd) == set(rsd)
    assert all(tuple(sd[k].shape) == tuple(rsd[k].shape) for k in sd)
    assert tuple(sd["conv_in.weight"].shape) == (320, 9, 3, 3) and tuple(sd["conv_out.weight"].shape) == (4, 320, 3, 3)
    assert sum(p.numel() for p in m.parameters()) == 859_535_364 == 859_520_964 + 320 * 5 * 9
    assert m.in_channels == 9 and m.config.out_channels == 4


def test_nine_channel_unet_loads_oracle_strict_and_refuses_training():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES, make_oracle_unet
    oracle = make_oracle_unet(seed=0, in_channels=9, **TINY_OVERRIDES)
    m = UNet2DConditionModel(in_channels=9, **TINY_OVERRIDES)
    m.load_state_dict(oracle.state_dict(), strict=True)
    assert torch.equal(m.conv_in.weight, oracle.conv_in.weight)
    x = torch.randn(2, 9, 16, 16, requires_grad=True)
    with pytest.raises(NotImplementedError):     # raised before anything reaches a device
        m(x, 10, torch.randn(2, 77, 64))


def _pipe(in_channels, cls_name="StableDiffusionInpaintPipeline"):
    import b200sd
    from b200sd.schedulers import DDIMScheduler
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import TINY_OVERRIDES
    unet = UNet2DConditionModel(in_channels=in_channels, **TINY_OVERRIDES)
    return getattr(b200sd, cls_name)(vae=object(), unet=unet.eval(), scheduler=DDIMScheduler(**_KW, clip_sample=False))


def test_inpaint_pipeline_argument_errors():
    image, mask = _pil_pair(64, 64)
    ctx2 = torch.zeros(2, 77, 64)
    with pytest.raises(ValueError, match="9"):
        _pipe(4)(prompt_embeds=ctx2, image=image, mask_image=mask, height=64, width=64)
    pipe = _pipe(9)
    with pytest.raises(ValueError, match="height x width"):          # the image is not resized
        pipe(prompt_embeds=ctx2, image=image, mask_image=mask, height=64, width=128)
    with pytest.raises(ValueError, match="mask_image"):
        pipe(prompt_embeds=ctx2, image=image, mask_image=_pil_pair(64, 56)[1], height=64, width=64)
    with pytest.raises(ValueError, match="image must be"):
        pipe(prompt_embeds=ctx2, image=torch.zeros(1, 3, 64, 72), mask_image=torch.zeros(1, 1, 64, 72), height=64, width=64)
    with pytest.raises(ValueError, match="batch"):
        pipe(prompt_embeds=ctx2, image=torch.zeros(3, 3, 64, 64), mask_image=torch.zeros(1, 1, 64, 64), height=64, width=64)
    with pytest.raises(ValueError, match="divisible"):
        pipe(prompt_embeds=ctx2, image=image, mask_image=mask, height=60, width=64)
    for kw in (dict(num_images_per_prompt=2), dict(callback=print)):
        with pytest.raises(TypeError):
            pipe(prompt_embeds=ctx2, image=image, mask_image=mask, height=64, width=64, **kw)


@pytest.mark.parametrize("cls_name", ["StableDiffusionPipeline", "StableDiffusionImg2ImgPipeline",
                                      "StableDiffusionInpaintPipelineLegacy"])
def test_four_channel_pipelines_refuse_the_nine_channel_unet(cls_name):
    pipe = _pipe(9, cls_name)
    ctx2 = torch.zeros(2, 77, 64)
    kw = dict(height=64, width=64) if cls_name == "StableDiffusionPipeline" else dict(init_image=torch.zeros(1, 3, 64, 64))
    if cls_name.endswith("Legacy"):
        kw["mask_image"] = torch.ones(1, 4, 8, 8)
    with pytest.raises(ValueError, match="StableDiffusionInpaintPipeline"):
        pipe(prompt_embeds=ctx2, **kw)


def test_denoise_loop_and_sampler_argument_errors():
    from b200sd.pipeline import denoise_loop
    from b200sd.sampler import CapturedSampler
    from b200sd.schedulers import DDIMScheduler
    pipe4, pipe9 = _pipe(4), _pipe(9)
    sch = DDIMScheduler(**_KW, clip_sample=False)
    lat, ctx2 = torch.zeros(1, 4, 8, 8), torch.zeros(2, 77, 64)
    with pytest.raises(ValueError, match="cond"):
        denoise_loop(pipe9.unet, sch, lat, ctx2, 2)                                 # 9 channels without cond
    with pytest.raises(ValueError, match="cond"):
        denoise_loop(pipe9.unet, sch, lat, ctx2, 2, cond=torch.zeros(1, 4, 8, 8))   # cond must hold 5 channels
    with pytest.raises(ValueError, match="no cond"):
        denoise_loop(pipe4.unet, sch, lat, ctx2, 2, cond=torch.zeros(1, 5, 8, 8))
    with pytest.raises(ValueError, match="full schedule"):
        denoise_loop(pipe9.unet, sch, lat, ctx2, 2, start=1, cond=torch.zeros(1, 5, 8, 8))
    sch.set_timesteps(10)
    for kw in (dict(start=3), dict(inpaint=True)):
        with pytest.raises(ValueError, match="full schedule"):
            CapturedSampler(pipe9.unet, sch, 1, 8, 8, 77, 7.5, **kw)


def test_saved_directory_loads_into_the_inpaint_class(tmp_path):
    from b200sd import StableDiffusionInpaintPipeline
    pipe = _pipe(9)
    pipe.vae = None
    with torch.no_grad():
        for p in pipe.unet.parameters():
            p.normal_()
    pipe.save_pretrained(str(tmp_path))
    index = json.load(open(tmp_path / "model_index.json"))
    assert index["_class_name"] == "StableDiffusionInpaintPipeline"
    assert json.load(open(tmp_path / "unet" / "config.json"))["in_channels"] == 9
    back = StableDiffusionInpaintPipeline.from_pretrained(str(tmp_path))
    assert type(back) is StableDiffusionInpaintPipeline and back.unet.in_channels == 9
    assert type(back.scheduler).__name__ == "DDIMScheduler"
    for (k, a), (k2, b) in zip(pipe.unet.state_dict().items(), back.unet.state_dict().items()):
        assert k == k2 and torch.equal(a, b)
