"""Caller of the hot path: ``get_latent_z`` / ``image_guided_synthesis`` (reference: utils/diffusion_utils.py:110-201) --
SURVEY.md 8(f) rank f2.

Same signature, conditioning construction, RNG order and return layout (``[batch, n_samples, c, t, h, w]``) as the
reference function, which ``viewcrafter.py:run_diffusion`` (viewcrafter.py:92-107) calls once per clip.  ``model`` is the
reference's ``VIPLatentDiffusion`` (with the U-Net / VAE / image_proj_model swapped for the viewcrafter_b200 classes by the
YAML ``target:`` lines, INTEGRATION.md) or any object with the same attributes: ``embedder``, ``image_proj_model``,
``get_learned_conditioning``, ``encode_first_stage``, ``decode_first_stage``, ``uncond_type``, ``model.conditioning_key``.

What differs from the reference, all parity-preserving (SURVEY.md App. C):
  * the sampler is created with ``batch_cfg=True``: cond + uncond run as one B=2 U-Net forward with the context-free prefix
    computed once, and -- because the same ``cond`` / ``uc`` tensors are handed to every step and every ``n_samples``
    iteration -- the cross-attention K/V projections are computed once per clip;
  * ``cuda_graph=True`` lets the viewcrafter_b200 U-Net replay its forward as one captured CUDA graph from the third call on
    (``UNetModel.enable_cuda_graph``): same kernels in the same order, ~1000 launches -> 1 per forward;
  * under ``parallel.shard_model`` the VAE encode and decode are split by frame over all ranks (``parallel.vae_encode_sharded`` /
    ``vae_decode_sharded``), with the posterior draws still taken in the reference's order on every rank;
  * nothing else: conditioning tensors, ``x_T`` / per-step noise draws and the decode are the reference's, in its order.
"""
from __future__ import annotations

import torch

from . import parallel
from .ddim import DDIMSampler
from .ddim_multiplecond import DDIMSampler as DDIMSampler_multicond


def get_latent_z(model, videos):
    """videos [b, c, t, h, w] -> latents [b, c', t, h/8, w/8] via per-frame encode_first_stage (diffusion_utils.py:110-115).
    Under parallel.shard_model the frames are encoded on all ranks (parallel.vae_encode_sharded): same result, same RNG draws."""
    if getattr(model, "_vae", None) is not None:
        return parallel.vae_encode_sharded(model, videos)
    b, c, t, h, w = videos.shape
    x = videos.permute(0, 2, 1, 3, 4).reshape(b * t, c, h, w)
    z = model.encode_first_stage(x)
    return z.reshape(b, t, *z.shape[1:]).permute(0, 2, 1, 3, 4)


@torch.no_grad()
def image_guided_synthesis(model, prompts, videos, noise_shape, n_samples=1, ddim_steps=50, ddim_eta=1.,
                           unconditional_guidance_scale=1.0, cfg_img=None, fs=None, text_input=False, multiple_cond_cfg=False,
                           timestep_spacing='uniform', guidance_rescale=0.0, condition_index=None, batch_cfg=True, cuda_graph=True,
                           **kwargs):
    unet = getattr(getattr(model, "model", None), "diffusion_model", None)
    if cuda_graph and hasattr(unet, "enable_cuda_graph") and next(unet.parameters()).is_cuda:
        unet.enable_cuda_graph()              # the ~100 forwards of a clip share shapes, weights and context: capture once, replay
    ddim_sampler = DDIMSampler(model, batch_cfg=batch_cfg) if not multiple_cond_cfg else DDIMSampler_multicond(model, batch_cfg=batch_cfg)
    batch_size = noise_shape[0]
    fs = torch.tensor([fs] * batch_size, dtype=torch.long, device=model.device)

    if not text_input:
        prompts = [""] * batch_size
    assert condition_index is not None, "Error: condition index is None!"

    img = videos[:, :, condition_index[0]]                                   # b c h w
    img_emb = model.image_proj_model(model.embedder(img))                   # b l c
    cond_emb = model.get_learned_conditioning(prompts)
    cond = {"c_crossattn": [torch.cat([cond_emb, img_emb], dim=1)]}
    hybrid = model.model.conditioning_key == 'hybrid'
    if hybrid:
        img_cat_cond = get_latent_z(model, videos)                           # b c t h w
        cond["c_concat"] = [img_cat_cond]

    uc = None
    if unconditional_guidance_scale != 1.0:
        if model.uncond_type == "empty_seq":
            uc_emb = model.get_learned_conditioning(batch_size * [""])
        elif model.uncond_type == "zero_embed":
            uc_emb = torch.zeros_like(cond_emb)
        else:
            raise ValueError(f"unknown uncond_type {model.uncond_type!r}")
        uc_img_emb = model.image_proj_model(model.embedder(torch.zeros_like(img)))
        uc = {"c_crossattn": [torch.cat([uc_emb, uc_img_emb], dim=1)]}
        if hybrid:
            uc["c_concat"] = [img_cat_cond]                                  # the SAME tensor as cond's: enables the shared CFG prefix

    # one more unconditional branch for the three-way CFG: image kept, text dropped (diffusion_utils.py:157-165)
    if multiple_cond_cfg and cfg_img != 1.0:
        uc_2 = {"c_crossattn": [torch.cat([uc_emb, img_emb], dim=1)]}
        if hybrid:
            uc_2["c_concat"] = [img_cat_cond]
        kwargs.update({"unconditional_conditioning_img_nonetext": uc_2})
    else:
        kwargs.update({"unconditional_conditioning_img_nonetext": None})

    batch_variants = []
    for _ in range(n_samples):
        samples, _ = ddim_sampler.sample(S=ddim_steps, conditioning=cond, batch_size=batch_size, shape=noise_shape[1:], verbose=False,
                                         unconditional_guidance_scale=unconditional_guidance_scale, unconditional_conditioning=uc,
                                         eta=ddim_eta, cfg_img=cfg_img, mask=None, x0=None, fs=fs,
                                         timestep_spacing=timestep_spacing, guidance_rescale=guidance_rescale, **kwargs)
        # latent -> pixel space; under parallel.shard_model every rank decodes its frames and gathers the rest
        sharded = getattr(model, "_vae", None) is not None
        batch_variants.append(parallel.vae_decode_sharded(model, samples) if sharded else model.decode_first_stage(samples))
    return torch.stack(batch_variants).permute(1, 0, 2, 3, 4, 5)              # batch, variants, c, t, h, w
