"""ORACLE (test infrastructure): the parity cases shared by the golden-vector generator (real reference classes
through the diffusers shim), the oracle self-check and the GPU parity tests.  Every input is produced by
oracle.weights.seeded_tensor so the three parties see identical values."""
from __future__ import annotations

import torch

from .weights import seeded_tensor


def to_double(x):
    """Floating-point tensors of a (nested) inputs structure in float64; everything else unchanged."""
    if torch.is_tensor(x):
        return x.double() if x.is_floating_point() else x
    if isinstance(x, (list, tuple)):
        return type(x)(to_double(v) for v in x)
    if isinstance(x, dict):
        return {k: to_double(v) for k, v in x.items()}
    return x

# residual shapes of the SD1.5 ControlNet for a base (latent) resolution r: 12 down tensors + mid
CN_CHANNELS = [320, 320, 320, 320, 640, 640, 640, 1280, 1280, 1280, 1280, 1280]
CN_DIV = [1, 1, 1, 2, 2, 2, 4, 4, 4, 8, 8, 8]


def controlnet_residuals(n: int, r: int, seed: int = 0):
    down = [seeded_tensor(f"down{i}", (n, c, max(r // d, 1), max(r // d, 1)), seed) for i, (c, d) in
            enumerate(zip(CN_CHANNELS, CN_DIV))]
    mid = seeded_tensor("mid", (n, 1280, max(r // 8, 1), max(r // 8, 1)), seed)
    return down, mid


ADAPTER_SDXL_KW = dict(backbone_model_name="sdxl", num_blocks=1, num_frames=1, num_adapters_per_location=3,
                       cross_attention_dim=2048, add_spatial_resnet=True, add_temporal_resnet=False,
                       add_spatial_transformer=True, add_temporal_transformer=False, add_adapter_location_A=True,
                       add_adapter_location_B=True, add_adapter_location_C=True)  # configs/sdxl_train_depth.yaml:40-54

ADAPTER_VIDEO_KW = dict(backbone_model_name="i2vgenxl", num_blocks=1, num_frames=4, num_adapters_per_location=3,
                        cross_attention_dim=1024, add_spatial_resnet=True, add_temporal_resnet=True,
                        add_spatial_transformer=True, add_temporal_transformer=True, add_adapter_location_A=True,
                        add_adapter_location_B=True, add_adapter_location_C=True, add_adapter_location_D=True,
                        add_adapter_location_M=True)  # configs/i2vgenxl_train_depth.yaml


def adapter_sdxl_inputs(n: int = 2, r: int = 8, seed: int = 0):
    down, _ = controlnet_residuals(n, r, seed)
    ctx = seeded_tensor("prompt_embeds", (n, 77, 2048), seed)
    return dict(down_block_res_samples=down, mid_block_res_sample=None, num_frames=1, timestep=torch.tensor(981.0),
                encoder_hidden_states=ctx)


def adapter_video_inputs(b: int = 1, f: int = 4, r: int = 8, seed: int = 0):
    down, mid = controlnet_residuals(b * f, r, seed)
    ctx = seeded_tensor("image_embeddings", (1, 1, 1024), seed)
    return dict(down_block_res_samples=down, mid_block_res_sample=mid, num_frames=f, timestep=torch.tensor(501.0),
                encoder_hidden_states=ctx)


CONTROLNET_KW = dict(cross_attention_dim=768)  # lllyasviel/control_v11*_sd15_* (SD1.5) configuration


def controlnet_inputs(n: int = 2, r: int = 8, seed: int = 0):
    return dict(sample=seeded_tensor("cn_sample", (n, 4, r, r), seed), timestep=torch.tensor(961.0),
                encoder_hidden_states=seeded_tensor("cn_ehs", (n, 77, 768), seed),
                controlnet_cond=torch.sigmoid(seeded_tensor("cn_cond", (n, 3, 8 * r, 8 * r), seed)),
                conditioning_scale=1.0, return_dict=False)


ROUTER_KW = dict(num_experts=7, backbone_model_name="i2vgenxl", router_type="simple_weights", num_routers=12,
                 add_mid_block_router=True)
ROUTER_MASK = [1, 1, 0, 1, 0, 0, 0]  # inference.py:343-345 for control types [depth, canny, softedge]


def unet_sdxl_inputs(n: int = 2, r: int = 16, seed: int = 0, with_residuals: bool = True):
    """r = UNet latent resolution; adapter residuals follow the 9 SDXL skip shapes."""
    chans = [320, 320, 320, 320, 640, 640, 640, 1280, 1280]
    divs = [1, 1, 1, 2, 2, 2, 4, 4, 4]
    res = [seeded_tensor(f"unet_res{i}", (n, c, r // d, r // d), seed, 0.5) for i, (c, d) in enumerate(zip(chans, divs))]
    res += [torch.zeros(n, 1280, r // 4, r // 4)] * 3  # the adapter returns 12 tensors; zip() drops the last 3
    return dict(sample=seeded_tensor("unet_sample", (n, 4, r, r), seed), timestep=torch.tensor(961.0),
                encoder_hidden_states=seeded_tensor("unet_ehs", (n, 77, 2048), seed),
                added_cond_kwargs=dict(text_embeds=seeded_tensor("unet_text_embeds", (n, 1280), seed),
                                       time_ids=torch.tensor([[8.0 * r, 8.0 * r, 0, 0, 8.0 * r, 8.0 * r]] * n)),
                down_block_additional_residuals=res if with_residuals else None,
                mid_block_additional_residual=0 if with_residuals else None)


def unet_i2vgen_inputs(b: int = 1, f: int = 4, r: int = 16, seed: int = 0, with_residuals: bool = True):
    """I2VGen-XL UNet inputs: sample (b,4,f,r,r), image_latents (b,4,f,r,r), image_embeddings (b,1024) -- the pipeline
    passes (2,1,1024) and `.view(-1, 4, 1024)` flattens it --, text states (b,77,1024), fps (b,)."""
    res = mid = None
    if with_residuals:
        down, mid = controlnet_residuals(b * f, r, seed)
        res = [d * 0.5 for d in down]
        mid = mid * 0.5
    return dict(sample=seeded_tensor("i2v_sample", (b, 4, f, r, r), seed), timestep=torch.tensor(961.0),
                fps=torch.tensor([16.0] * b), image_latents=seeded_tensor("i2v_image_latents", (b, 4, f, r, r), seed),
                image_embeddings=seeded_tensor("i2v_image_embeddings", (b, 1, 1024), seed),
                encoder_hidden_states=seeded_tensor("i2v_ehs", (b, 77, 1024), seed),
                down_block_additional_residuals=res, mid_block_additional_residual=mid)


# Reduced-width configurations of the two video UNets: same block types, depths and code paths as the released models
# (block_out_channels 320/640/1280/1280), small enough that the REAL reference classes run on CPU in seconds when the
# golden vectors are generated (tests/golden/make_golden.py) and checked (tests/test_oracle_golden.py).
UNET_SVD_SMALL_KW = dict(in_channels=8, out_channels=4, block_out_channels=(64, 128, 256, 256),
                         num_attention_heads=(2, 4, 4, 8), cross_attention_dim=96, addition_time_embed_dim=32,
                         projection_class_embeddings_input_dim=96, layers_per_block=2, num_frames=4)
# released stable-video-diffusion-img2vid unet config.json (the reference class default has heads (5, 10, 10, 20))
UNET_SVD_KW = dict(num_attention_heads=(5, 10, 20, 20), num_frames=14)
UNET_I2VGEN_SMALL_KW = dict(in_channels=4, out_channels=4, block_out_channels=(64, 128, 256, 256), layers_per_block=2,
                            norm_num_groups=32, cross_attention_dim=96, attention_head_dim=32)


def unet_svd_inputs(b: int = 1, f: int = 4, r: int = 16, seed: int = 0, with_residuals: bool = True,
                    chans=(64, 128, 256, 256), ctx: int = 96):
    """SVD UNet inputs (svd/pipelines/svd_controlnet_adapter_pipeline.py call site): sample (b, f, 8, r, r), image
    embedding (b, 1, ctx), added_time_ids (b, 3) = [fps - 1, motion bucket, noise aug]; the adapter residuals are passed
    5-D ("b c f h w") with three surplus entries at the end (zip() truncation, quirk Q7) and a 5-D mid residual."""
    res = mid = None
    if with_residuals:
        c0, c1, c2, c3 = chans
        shapes = [(c0, 1), (c0, 1), (c0, 1), (c0, 2), (c1, 2), (c1, 2), (c1, 4), (c2, 4), (c2, 4), (c2, 8), (c3, 8),
                  (c3, 8)]
        res = [seeded_tensor(f"svd_res{i}", (b, c, f, r // d, r // d), seed, 0.5) for i, (c, d) in enumerate(shapes)]
        res += [torch.zeros(b, c3, f, r // 8, r // 8)] * 3
        mid = seeded_tensor("svd_mid", (b, c3, f, r // 8, r // 8), seed, 0.5)
    return dict(sample=seeded_tensor("svd_sample", (b, f, 8, r, r), seed), timestep=torch.tensor(1.6377),
                encoder_hidden_states=seeded_tensor("svd_ehs", (b, 1, ctx), seed),
                added_time_ids=torch.tensor([[6.0, 127.0, 0.02]] * b),
                down_block_additional_residuals=res, mid_block_additional_residual=mid)


def unet_i2vgen_small_inputs(b: int = 1, f: int = 4, r: int = 16, seed: int = 0, with_residuals: bool = True,
                             chans=(64, 128, 256, 256), ctx: int = 96):
    """Inputs of the reduced-width I2VGen-XL UNet (UNET_I2VGEN_SMALL_KW); residuals 4-D (b f) c h w as the pipeline
    passes them (i2vgen_xl/pipelines/...pipeline.py:1080-1082), 12 entries for 12 skip tensors."""
    res = mid = None
    c0, c1, c2, c3 = chans
    if with_residuals:
        shapes = [(c0, 1), (c0, 1), (c0, 1), (c0, 2), (c1, 2), (c1, 2), (c1, 4), (c2, 4), (c2, 4), (c2, 8), (c3, 8),
                  (c3, 8)]
        res = [seeded_tensor(f"i2vs_res{i}", (b * f, c, r // d, r // d), seed, 0.5) for i, (c, d) in enumerate(shapes)]
        mid = seeded_tensor("i2vs_mid", (b * f, c3, r // 8, r // 8), seed, 0.5)
    return dict(sample=seeded_tensor("i2vs_sample", (b, 4, f, r, r), seed), timestep=torch.tensor(961.0),
                fps=torch.tensor([16.0] * b), image_latents=seeded_tensor("i2vs_image_latents", (b, 4, f, r, r), seed),
                image_embeddings=seeded_tensor("i2vs_image_embeddings", (b, 1, ctx), seed),
                encoder_hidden_states=seeded_tensor("i2vs_ehs", (b, 77, ctx), seed),
                down_block_additional_residuals=res, mid_block_additional_residual=mid)
