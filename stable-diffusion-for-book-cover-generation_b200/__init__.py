"""b200sd -- B200-native (sm_100a) SD v1.x UNet denoise hot path behind the diffusers class surface.

Public surface (mirrors what finetune_sd.py / inference.py / StableDiffusionPipeline touch):
    UNet2DConditionModel, DDIMScheduler, PNDMScheduler, DDPMScheduler, StableDiffusionPipeline,
    StableDiffusionImg2ImgPipeline, StableDiffusionInpaintPipelineLegacy (image-to-image, legacy inpainting), denoise_loop, mse_loss,
    CapturedSampler (the whole denoising step as one CUDA graph), CLIPTextModel (transformers' surface, own kernels),
    AutoencoderKL (diffusers' surface, own kernels)
"""
__version__ = "0.1.0"


def __getattr__(name):  # lazy: importing the package must not require torch.cuda or the .so
    import importlib
    table = {
        "UNet2DConditionModel": "b200sd.unet",
        "DDIMScheduler": "b200sd.schedulers",
        "PNDMScheduler": "b200sd.schedulers",
        "DDPMScheduler": "b200sd.schedulers",
        "denoise_loop": "b200sd.pipeline",
        "StableDiffusionPipeline": "b200sd.pipeline",
        "StableDiffusionImg2ImgPipeline": "b200sd.pipeline",
        "StableDiffusionInpaintPipelineLegacy": "b200sd.pipeline",
        "mse_loss": "b200sd.ops",
        "CapturedSampler": "b200sd.sampler",
        "CLIPTextModel": "b200sd.clip",
        "CLIPTextConfig": "b200sd.clip",
        "AutoencoderKL": "b200sd.vae",
    }
    if name in table:
        return getattr(importlib.import_module(table[name]), name)
    raise AttributeError(name)
