"""Drop-in ``DDIMSampler`` with three-way classifier-free guidance (reference: lvdm/models/samplers/ddim_multiplecond.py),
the sampler ``image_guided_synthesis(..., multiple_cond_cfg=True)`` selects (utils/diffusion_utils.py:9,119).

Differences from ``viewcrafter_b200.ddim.DDIMSampler`` -- exactly the reference's:
  * three ``apply_model`` calls per step: cond, uncond and ``unconditional_conditioning_img_nonetext`` (image kept, text
    dropped), combined as ``u + cfg_img (v_img - u) + s (v_cond - v_img)`` (ddim_multiplecond.py:227-233);
    ``cfg_img`` defaults to the text scale;
  * ``ddim_scale_arr_prev[0] = ddim_scale_arr[0]`` (ddim_multiplecond.py:33; ddim.py:33-35 fixed this one only), so the last
    step's dynamic rescale differs between the two samplers (SURVEY.md App. D).
The combine, guidance rescale, v->(eps, x0), dynamic rescale and x_{t-1} are one fused CUDA update (vc_ddim_update3).

How the three predictions are computed (same values as three separate calls, see _apply_three):
  * ``batch_cfg=True`` with stackable conditioning: ONE U-Net forward at B=3 (cond, uncond, image-only) whose context-free
    prefix runs once when the three branches share x and c_concat (one GPU, or pure frame sharding: B=3 per rank);
  * under the CFG rank split of ``parallel.shard_model``: the branch-0 ranks run (cond, image-only) as one B=2 forward, the
    branch-1 ranks uncond at B=1, and ``CfgComm.exchange3`` hands every rank all three;
  * otherwise the reference's separate calls.
"""
from __future__ import annotations

import torch

from . import ops
from .ddim import DDIMSampler as _TwoWaySampler
from .unet import SHARED_PREFIX_ANY_LAYOUT


class DDIMSampler(_TwoWaySampler):
    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0., verbose=True):
        super().make_schedule(ddim_num_steps, ddim_discretize, ddim_eta, verbose)
        if self.use_dynamic_rescale:
            self.ddim_scale_arr_prev = torch.cat([self.ddim_scale_arr[0:1], self.ddim_scale_arr[:-1]])

    @torch.no_grad()
    def p_sample_ddim(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                      temperature=1., noise_dropout=0., score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1., unconditional_conditioning=None, uc_type=None, cfg_img=None,
                      mask=None, x0=None, guidance_rescale=0.0, _step=None, **kwargs):
        self._check_step_options(use_original_steps, quantize_denoised, score_corrector)
        if cfg_img is None:
            cfg_img = unconditional_guidance_scale
        uc_img = kwargs['unconditional_conditioning_img_nonetext']           # KeyError like ddim_multiplecond.py:224
        step = int(t[0].item()) if _step is None else _step
        v_u = v_i = None
        if unconditional_conditioning is None or unconditional_guidance_scale == 1.:
            v_c = self.model.apply_model(x, t, c, **kwargs)
        else:
            if uc_img is None:
                raise ValueError("three-way CFG needs unconditional_conditioning_img_nonetext (image_guided_synthesis only builds it "
                                 "when cfg_img != 1.0, utils/diffusion_utils.py:157-163)")
            v_c, v_u, v_i = self._apply_three(x, t, c, unconditional_conditioning, uc_img, kwargs)
        sc = self.step_scalars(index, step)
        sc["cfg_scale"], sc["guidance_rescale"] = float(unconditional_guidance_scale), float(guidance_rescale)
        noise = self._step_noise(x, repeat_noise, temperature, noise_dropout)
        return self._fused_update(x, v_c, v_u, noise, sc, v_uncond_img=v_i, cfg_img=float(cfg_img))

    @staticmethod
    def _stackable(conds):
        return all(isinstance(d, dict) for d in conds) and all(d.keys() == conds[0].keys() for d in conds)

    def _apply_stacked(self, x, t, conds, kwargs):
        """The branches of `conds` as ONE forward at B = len(conds) * x.shape[0], stacked in the given order with the tensors built
        once per set of dicts (so that the U-Net's K/V cache and captured graph hit every step).  Returns one prediction per dict."""
        n, k = x.shape[0], len(conds)
        cat, same_concat = self._stack_conditionings(conds)
        kw = {key: (torch.cat([v] * k, 0) if isinstance(v, torch.Tensor) and v.dim() >= 1 and v.shape[0] == n else v)
              for key, v in kwargs.items()}
        if same_concat and n == 1:
            # every branch sees the same x, t, fs and c_concat: the U-Net computes the context-free prefix once, also when it is
            # frame-sharded (ignored by models that do not know the hint)
            kw["cfg_shared_prefix"] = SHARED_PREFIX_ANY_LAYOUT
        out = self.model.apply_model(torch.cat([x] * k, 0), torch.cat([t] * k, 0), cat, **kw)
        return [out[i * n:(i + 1) * n].contiguous() for i in range(k)]

    def _apply_three(self, x, t, c, uc, uc_img, kwargs):
        """(v_cond, v_uncond, v_img) of one step."""
        cfg = getattr(self.model, "_cfg", None)
        if cfg is not None:                     # multi-GPU CFG split: branch 0 computes (cond, image-only), branch 1 uncond
            if cfg.branch == 0:
                pair = [c, uc_img]
                v_c, v_i = self._apply_stacked(x, t, pair, kwargs) if self._stackable(pair) else \
                    (self.model.apply_model(x, t, c, **kwargs), self.model.apply_model(x, t, uc_img, **kwargs))
                return cfg.exchange3(v_c.float().contiguous(), v_i.float().contiguous())
            return cfg.exchange3(self.model.apply_model(x, t, uc, **kwargs).float().contiguous())
        if self.batch_cfg and self._stackable([c, uc, uc_img]):
            return tuple(self._apply_stacked(x, t, [c, uc, uc_img], kwargs))
        v_c, v_u = self._apply_both(x, t, c, uc, kwargs)
        return v_c, v_u, self.model.apply_model(x, t, uc_img, **kwargs)
