"""The drop-in claim, end to end, against outputs of the UNMODIFIED reference pipeline (tests/golden/dropin_pipeline.npz,
written by oracle/make_golden.py):

the reference ran its own ``VIPLatentDiffusion``, instantiated from its own YAML (configs/inference_pvd_1024.yaml, reduced
widths), and its own ``utils.diffusion_utils.image_guided_synthesis`` with its own samplers, on weights synthesised from the
stored (name, shape) list.  Here the U-Net, AutoencoderKL and Resampler of viewcrafter_b200 are built from the constructor
arguments the YAML gave the reference's classes, must carry the same state-dict keys and shapes in the same order, get the
same weights, and run through viewcrafter_b200's ``LatentDiffusion`` wrapper, samplers and ``image_guided_synthesis`` with
the same arguments and seeds.  The CUDA ops are replaced by the torch double, so this checks every seam of the boundary
(constructor kwargs, state-dict keys, conditioning construction, RNG order, decode), not the kernels.  The two OpenCLIP
towers are the toys of oracle/synth.py on both sides.  T = 16 so that the per-frame image-token context branch
(openaimodel3d.py:556-560) is exercised, T = 5 for the shared-context branch of the 25-frame checkpoints.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import synth
from tests import fake_ops

NETS = ("model.", "first_stage_model.", "image_proj_model.")


def _model(gd):
    from viewcrafter_b200.diffusion import LatentDiffusion
    from viewcrafter_b200.resampler import Resampler

    class Model(LatentDiffusion):                         # the attribute surface image_guided_synthesis reads (synthesis.py)
        def __init__(self, P):
            super().__init__(json.loads(str(gd["unet_config"])), json.loads(str(gd["first_stage_config"])),
                             **{k: P[k] for k in ("timesteps", "linear_start", "linear_end", "rescale_betas_zero_snr", "parameterization",
                                                  "scale_factor", "use_dynamic_rescale", "base_scale", "perframe_ae", "conditioning_key")})
            self.uncond_type = P["uncond_type"]
            self.cond_stage_model = synth.ToyText()
            self.embedder = synth.ToyImage()
            self.image_proj_model = Resampler(**json.loads(str(gd["image_proj_config"])))

        def get_learned_conditioning(self, c):
            return self.cond_stage_model.encode(c)

    torch.manual_seed(0)
    return Model(json.loads(str(gd["model_params"]))).eval()


@pytest.mark.parametrize("multi,T", [(False, 16), (True, 16), (False, 5)])
def test_reference_pipeline_with_dropins_matches_reference(monkeypatch, golden_dir, multi, T):
    """T = 16: 77 + 16 T = 333 context tokens -> per-frame image tokens (openaimodel3d.py:556-560); T = 5: the
    shared-context branch the 25-frame checkpoints take."""
    from viewcrafter_b200.synthesis import image_guided_synthesis
    fake_ops.install(monkeypatch)
    gd = np.load(os.path.join(golden_dir, "dropin_pipeline.npz"))
    tag = f"multi{int(multi)}_T{T}"
    mine = _model(gd)
    ref_shapes = [(n, tuple(s)) for n, s in json.loads(str(gd["shapes"]))]
    assert [(k, s) for k, s in synth.module_shapes(mine) if k.startswith(NETS)] == ref_shapes     # names, shapes AND order
    sd = mine.state_dict()
    sd.update(synth.synth_state_dict(ref_shapes, seed=81))
    mine.load_state_dict(sd, strict=True)

    H, W = 8, 8
    videos = torch.rand(1, 3, T, 8 * H, 8 * W, generator=torch.Generator().manual_seed(7)) * 2 - 1
    kw = json.loads(str(gd[f"{tag}_kwargs"]))
    torch.manual_seed(11)
    out = image_guided_synthesis(mine, ["a photo"], videos, [1, 4, T, H, W], **kw)
    assert tuple(out.shape) == tuple(gd[f"{tag}_shape"]) == (1, 1, 3, T, 8 * H, 8 * W) and out.dtype == torch.float32
    ref = torch.from_numpy(gd[f"{tag}_sample"])
    err = (out.reshape(-1)[::int(gd["stride"])] - ref).abs()
    std = float(gd[f"{tag}_std"])
    # fp16 rounding points of the kernels (emulated by the op double) vs the fp32 reference, amplified ~16x by CFG 7.5 per step
    assert float(err.mean()) < 0.03 * std and float(err.max()) < 0.35 * std, (float(err.mean()), float(err.max()), std)
