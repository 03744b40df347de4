"""Import the UNMODIFIED reference modules from a checkout of the reference (VC_REFERENCE_ROOT).

TEST INFRASTRUCTURE.  Used by oracle/make_golden.py to write tests/golden/; the tests only read
those fixtures.  Never imported by the product.

Shims (SURVEY.md §8c): a stub ``pytorch_lightning`` package (the reference only uses it as a
base class), and on CPU an override of ``DDIMSampler.register_buffer`` because
lvdm/models/samplers/ddim.py:18-22 hard-codes "cuda".
"""
from __future__ import annotations

import os
import sys
import types

import torch

REF_ROOT = os.environ.get("VC_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "lvdm"))


def install():
    if not available():
        raise RuntimeError(f"reference not found at {REF_ROOT}")
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")

        class LightningModule(torch.nn.Module):
            @property
            def device(self):
                try:
                    return next(self.parameters()).device
                except StopIteration:
                    return torch.device("cpu")

            def log(self, *a, **k):
                pass

            def log_dict(self, *a, **k):
                pass

        pl.LightningModule = LightningModule
        pl.seed_everything = lambda s: torch.manual_seed(s)
        util = types.ModuleType("pytorch_lightning.utilities")
        util.rank_zero_only = lambda f: f
        pl.utilities = util
        sys.modules["pytorch_lightning"] = pl
        sys.modules["pytorch_lightning.utilities"] = util
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)


UNET_KW = dict(in_channels=8, out_channels=4, model_channels=320, attention_resolutions=[4, 2, 1],
               num_res_blocks=2, channel_mult=[1, 2, 4, 4], dropout=0.1, num_head_channels=64,
               transformer_depth=1, context_dim=1024, use_linear=True, use_checkpoint=False,
               temporal_conv=True, temporal_attention=True, temporal_selfatt_only=True,
               use_relative_position=False, use_causal_attention=False, temporal_length=16,
               addition_attention=True, image_cross_attention=True, default_fs=10, fs_condition=True)

VAE_DD = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
              ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0)


def randomize_zero_params(module: torch.nn.Module, seed: int = 1, std: float = 0.02):
    """SURVEY.md §7 'hard parts': zero-initialised tensors make parity vacuous; redraw them."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for _, p in sorted(module.named_parameters()):
            if p.numel() > 0 and float(p.abs().max()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g) * std)


def build_unet(seed=0, **over):
    install()
    from lvdm.modules.networks.openaimodel3d import UNetModel
    kw = dict(UNET_KW); kw.update(over)
    torch.manual_seed(seed)
    m = UNetModel(**kw).eval()
    randomize_zero_params(m)
    return m


def build_encoder(seed=0, **over):
    """Returns (encoder, quant_conv) as the reference AutoencoderKL builds them (autoencoder.py:28-32)."""
    install()
    from lvdm.modules.networks.ae_modules import Encoder
    dd = dict(VAE_DD); dd.update(over)
    torch.manual_seed(seed)
    enc = Encoder(**dd).eval()
    qc = torch.nn.Conv2d(2 * dd["z_channels"], 2 * 4, 1)
    return enc, qc


def build_decoder(seed=0, **over):
    """Returns (decoder, post_quant_conv) as the reference AutoencoderKL builds them (autoencoder.py:28-33)."""
    install()
    from lvdm.modules.networks.ae_modules import Decoder
    dd = dict(VAE_DD); dd.update(over)
    torch.manual_seed(seed)
    dec = Decoder(**dd).eval()
    pq = torch.nn.Conv2d(4, dd["z_channels"], 1)
    return dec, pq


RESAMPLER_KW = dict(dim=1024, depth=4, dim_head=64, heads=12, num_queries=16, embedding_dim=1280, output_dim=1024,
                    ff_mult=4, video_length=16)          # configs/inference_pvd_1024.yaml:100-111


def build_resampler(seed=0, **over):
    """The unmodified reference Resampler (image_proj_model, ddpm3d.py:1038-1039)."""
    install()
    from lvdm.modules.encoders.resampler import Resampler
    kw = dict(RESAMPLER_KW); kw.update(over)
    torch.manual_seed(seed)
    return Resampler(**kw).eval()
