"""Drop-in ``DDIMSampler`` (reference: lvdm/models/samplers/ddim.py:10-281).

Same constructor, ``make_schedule`` / ``sample`` / ``ddim_sampling`` / ``p_sample_ddim`` signatures and return values
(``(samples, {'x_inter': [...], 'pred_x0': [...]})``).  Host logic (schedule tables, loop, RNG draws with the same
shapes in the same order) is Python; everything after the two ``apply_model`` calls of a step -- CFG combine,
guidance rescale (two global unbiased stds), v->(eps, x0), dynamic rescale, x_{t-1} -- is ONE fused CUDA update
(vc_ddim_update).  ``batch_cfg=True`` runs cond+uncond as a single B=2 U-Net forward.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops, schedule


class DDIMSampler(object):
    def __init__(self, model, schedule="linear", batch_cfg: bool = False, **kwargs):
        super().__init__()
        self.model = model
        self.ddpm_num_timesteps = model.num_timesteps
        self.schedule = schedule
        self.counter = 0
        self.batch_cfg = batch_cfg

    def register_buffer(self, name, attr):
        if isinstance(attr, torch.Tensor) and attr.device != self._device():
            attr = attr.to(self._device())
        setattr(self, name, attr)

    def _device(self):
        return self.model.betas.device

    def make_schedule(self, ddim_num_steps, ddim_discretize="uniform", ddim_eta=0., verbose=True):
        m = self.model
        self.ddim_timesteps = schedule.ddim_timesteps(ddim_discretize, ddim_num_steps, self.ddpm_num_timesteps)
        ac = m.alphas_cumprod
        assert ac.shape[0] == self.ddpm_num_timesteps, 'alphas have to be defined for each timestep'
        ac_cpu = ac.detach().to(torch.float32).cpu()
        self.use_dynamic_rescale = bool(getattr(m, "use_dynamic_rescale", False))
        if self.use_dynamic_rescale:
            arr = m.scale_arr.detach().float().cpu()
            self.ddim_scale_arr = arr[self.ddim_timesteps]
            self.ddim_scale_arr_prev = torch.cat([arr[0:1], self.ddim_scale_arr[:-1]])
        f32dev = lambda x: x.clone().detach().to(torch.float32).to(self._device())
        self.register_buffer('betas', f32dev(m.betas))
        self.register_buffer('alphas_cumprod', f32dev(ac))
        self.register_buffer('alphas_cumprod_prev', f32dev(m.alphas_cumprod_prev))
        self.register_buffer('sqrt_alphas_cumprod', f32dev(torch.sqrt(ac_cpu)))
        self.register_buffer('sqrt_one_minus_alphas_cumprod', f32dev(torch.sqrt(1. - ac_cpu)))
        sigmas, alphas, alphas_prev = schedule.ddim_parameters(ac_cpu, self.ddim_timesteps, ddim_eta)
        self.ddim_sigmas, self.ddim_alphas, self.ddim_alphas_prev = sigmas, alphas, alphas_prev
        self.ddim_sqrt_one_minus_alphas = np.sqrt(1. - alphas)
        # host copies of the model tables gathered by timestep t in the v-parameterisation (ddpm3d.py:239-251)
        self._sqrt_ac = m.sqrt_alphas_cumprod.detach().float().cpu()
        self._sqrt_1mac = m.sqrt_one_minus_alphas_cumprod.detach().float().cpu()
        if verbose:
            print(f'Selected timesteps for ddim sampler: {self.ddim_timesteps}')

    def step_scalars(self, index: int, step: int) -> dict:
        """The per-step fp32 scalars exactly as p_sample_ddim materialises them with torch.full (ddim.py:253-266)."""
        r = schedule.f32
        d = dict(a_t=r(self.ddim_alphas[index]), a_prev=r(self.ddim_alphas_prev[index]), sigma_t=r(self.ddim_sigmas[index]),
                 sqrt_one_minus_at=r(self.ddim_sqrt_one_minus_alphas[index]),
                 sqrt_ac_t=float(self._sqrt_ac[step]), sqrt_1mac_t=float(self._sqrt_1mac[step]))
        if self.use_dynamic_rescale:
            d["scale_t"], d["prev_scale_t"] = r(self.ddim_scale_arr[index]), r(self.ddim_scale_arr_prev[index])
        else:
            d["scale_t"] = d["prev_scale_t"] = 1.0
        return d

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0., mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
               corrector_kwargs=None, verbose=True, schedule_verbose=False, x_T=None, log_every_t=100,
               unconditional_guidance_scale=1., unconditional_conditioning=None, precision=None, fs=None,
               timestep_spacing='uniform', guidance_rescale=0.0, **kwargs):
        if conditioning is not None:
            first = conditioning[list(conditioning.keys())[0]] if isinstance(conditioning, dict) else conditioning
            try:
                cbs = first.shape[0]
            except AttributeError:
                cbs = first[0].shape[0]
            if cbs != batch_size:
                print(f"Warning: Got {cbs} conditionings but batch-size is {batch_size}")
        self.make_schedule(ddim_num_steps=S, ddim_discretize=timestep_spacing, ddim_eta=eta, verbose=schedule_verbose)
        if len(shape) == 3:
            size = (batch_size, *shape)
        elif len(shape) == 4:
            size = (batch_size, *shape)
        else:
            raise ValueError(f"shape must be (C,H,W) or (C,T,H,W), got {shape}")
        return self.ddim_sampling(conditioning, size, callback=callback, img_callback=img_callback, quantize_denoised=quantize_x0,
                                  mask=mask, x0=x0, ddim_use_original_steps=False, noise_dropout=noise_dropout,
                                  temperature=temperature, score_corrector=score_corrector, corrector_kwargs=corrector_kwargs,
                                  x_T=x_T, log_every_t=log_every_t, unconditional_guidance_scale=unconditional_guidance_scale,
                                  unconditional_conditioning=unconditional_conditioning, verbose=verbose, precision=precision,
                                  fs=fs, guidance_rescale=guidance_rescale, **kwargs)

    @torch.no_grad()
    def ddim_sampling(self, cond, shape, x_T=None, ddim_use_original_steps=False, callback=None, timesteps=None,
                      quantize_denoised=False, mask=None, x0=None, img_callback=None, log_every_t=100, temperature=1.,
                      noise_dropout=0., score_corrector=None, corrector_kwargs=None, unconditional_guidance_scale=1.,
                      unconditional_conditioning=None, verbose=True, precision=None, fs=None, guidance_rescale=0.0, **kwargs):
        if ddim_use_original_steps:
            # the reference's own branch reads self.ddim_sigmas_for_original_num_steps, which its make_schedule never defines (ddim.py:248)
            raise NotImplementedError("viewcrafter_b200.DDIMSampler: ddim_use_original_steps is not implemented (it fails in the reference too)")
        device = self._device()
        b = shape[0]
        img = torch.randn(shape, device=device) if x_T is None else x_T
        if precision is not None and int(precision) == 16:
            img = img.to(dtype=torch.float16)               # ddim.py:154-156: only x_T is rounded; every later latent is fp32 again
        steps = self.ddim_timesteps
        if timesteps is not None:                           # ddim.py:160-162: the first `timesteps / S` share of the sub-sequence, minus one
            subset_end = int(min(timesteps / steps.shape[0], 1) * steps.shape[0]) - 1
            steps = steps[:subset_end]
        total = steps.shape[0]
        intermediates = {'x_inter': [img], 'pred_x0': [img]}
        clean_cond = kwargs.pop("clean_cond", False)
        for i, step in enumerate(np.flip(steps)):
            index = total - i - 1
            ts = torch.full((b,), int(step), device=device, dtype=torch.long)
            if mask is not None:                            # ddim.py:178-185: keep the (noised) original where mask == 1 (plain tensor math:
                assert x0 is not None                       # not on the ViewCrafter path, which passes mask=None)
                img_orig = x0 if clean_cond else self.model.q_sample(x0, ts)
                img = img_orig * mask + (1. - mask) * img
            img, pred_x0 = self.p_sample_ddim(img, cond, ts, index=index, quantize_denoised=quantize_denoised,
                                              temperature=temperature, noise_dropout=noise_dropout,
                                              score_corrector=score_corrector, corrector_kwargs=corrector_kwargs,
                                              unconditional_guidance_scale=unconditional_guidance_scale,
                                              unconditional_conditioning=unconditional_conditioning, mask=mask, x0=x0, fs=fs,
                                              guidance_rescale=guidance_rescale, _step=int(step), **kwargs)
            if callback:
                callback(i)
            if img_callback:
                img_callback(pred_x0, i)
            if index % log_every_t == 0 or index == total - 1:
                intermediates['x_inter'].append(img)
                intermediates['pred_x0'].append(pred_x0)
        return img, intermediates

    def _stacked_conditioning(self, c, uc):
        """cond|uncond conditioning stacked along the batch axis, built once per (c, uc) pair and reused for every step:
        the sampler passes the same dicts for all steps (ddim.py:150-160), and handing the U-Net the SAME context tensor
        each step lets it keep the cross-attention K/V projections (SURVEY.md App. C.1).  Also reports whether the
        c_concat entries of the two branches are the same tensors (utils/diffusion_utils.py:152-153)."""
        return self._stack_conditionings((c, uc))

    def _stack_conditionings(self, conds):
        """_stacked_conditioning for any number of conditioning dicts with the same keys (stacked in the given order)."""
        sig = [(a, ops.tensor_version(a)) for k in conds[0] for ent in zip(*(d[k] for d in conds)) for a in ent]
        cached = getattr(self, "_cat_cache", None)
        if cached is not None and cached[0] == len(conds) and len(cached[1]) == len(sig) and all(v is not None for _, v in sig) and all(
                a is a0 and v == v0 for (a, v), (a0, v0) in zip(sig, cached[1])):
            return cached[2], cached[3]
        cat = {k: [torch.cat(ent, 0) for ent in zip(*(d[k] for d in conds))] for k in conds[0]}
        same = all(all((a is e[0]) or (a.shape == e[0].shape and bool(torch.equal(a, e[0]))) for a in e[1:])
                   for e in zip(*(d.get("c_concat", []) for d in conds))) if "c_concat" in conds[0] else False
        self._cat_cache = (len(conds), sig, cat, same)
        return cat, same

    def _apply_both(self, x, t, c, uc, kwargs):
        """cond + uncond as one B=2 forward when every conditioning entry can be stacked; else two calls (ddim.py:223-224)."""
        cfg = getattr(self.model, "_cfg", None)
        if cfg is not None:                                   # multi-GPU CFG split: this rank computes one branch only
            mine = self.model.apply_model(x, t, c if cfg.branch == 0 else uc, **kwargs)
            return cfg.exchange(mine.float().contiguous())
        if self.batch_cfg and isinstance(c, dict) and isinstance(uc, dict) and c.keys() == uc.keys():
            cat, same_concat = self._stacked_conditioning(c, uc)
            kw = {k: (torch.cat([v, v], 0) if isinstance(v, torch.Tensor) and v.dim() >= 1 and v.shape[0] == x.shape[0] else v)
                  for k, v in kwargs.items()}
            if same_concat and x.shape[0] == 1:
                # both branches see the same x, t, fs and c_concat: let the U-Net compute the context-free prefix once
                # (SURVEY.md App. C.2; ignored by models that do not know the hint)
                kw["cfg_shared_prefix"] = True
            out = self.model.apply_model(torch.cat([x, x], 0), torch.cat([t, t], 0), cat, **kw)
            n = x.shape[0]
            return out[:n].contiguous(), out[n:].contiguous()
        return self.model.apply_model(x, t, c, **kwargs), self.model.apply_model(x, t, uc, **kwargs)

    @torch.no_grad()
    def p_sample_ddim(self, x, c, t, index, repeat_noise=False, use_original_steps=False, quantize_denoised=False,
                      temperature=1., noise_dropout=0., score_corrector=None, corrector_kwargs=None,
                      unconditional_guidance_scale=1., unconditional_conditioning=None, uc_type=None,
                      conditional_guidance_scale_temporal=None, mask=None, x0=None, guidance_rescale=0.0, _step=None, **kwargs):
        self._check_step_options(use_original_steps, quantize_denoised, score_corrector)
        step = int(t[0].item()) if _step is None else _step
        if unconditional_conditioning is None or unconditional_guidance_scale == 1.:
            v_c, v_u = self.model.apply_model(x, t, c, **kwargs), None
        else:
            if not isinstance(c, (torch.Tensor, dict)):
                raise NotImplementedError
            v_c, v_u = self._apply_both(x, t, c, unconditional_conditioning, kwargs)
        sc = self.step_scalars(index, step)
        sc["cfg_scale"], sc["guidance_rescale"] = float(unconditional_guidance_scale), float(guidance_rescale)
        noise = self._step_noise(x, repeat_noise, temperature, noise_dropout)
        return self._fused_update(x, v_c, v_u, noise, sc)

    # -- pieces shared with the three-way sampler (ddim_multiplecond.py) ------------------------------------------------
    def _check_step_options(self, use_original_steps, quantize_denoised, score_corrector):
        if use_original_steps:
            raise NotImplementedError("viewcrafter_b200.DDIMSampler: use_original_steps is not implemented (ddim.py:248 fails in the reference too)")
        if quantize_denoised:
            raise NotImplementedError("viewcrafter_b200.DDIMSampler: quantize_denoised needs a VQ first stage (first_stage_model.quantize); "
                                      "AutoencoderKL has none")
        if getattr(self.model, "parameterization", "v") != "v":
            raise NotImplementedError("viewcrafter_b200.DDIMSampler: only the v-parameterisation is implemented")
        if score_corrector is not None:
            raise AssertionError("not implemented")          # ddim.py:239-241 asserts parameterization == 'eps' before using a score corrector

    @staticmethod
    def _step_noise(x, repeat_noise, temperature, noise_dropout):
        """noise_like * temperature, then dropout (ddim.py:275-277; the scalar sigma_t is applied by the fused update, which commutes with both)."""
        shape = (1, *x.shape[1:]) if repeat_noise else x.shape
        noise = torch.randn(shape, device=x.device)                      # same draw as lvdm/common.py:31-34
        if repeat_noise:
            noise = noise.repeat(x.shape[0], *((1,) * (x.dim() - 1)))
        if temperature != 1.:
            noise = noise * temperature
        if noise_dropout > 0.:
            noise = torch.nn.functional.dropout(noise, p=noise_dropout)
        return noise.contiguous()

    @staticmethod
    def _fused_update(x, v_c, v_u, noise, sc, **extra):
        """One fused update for the batch; the guidance rescale uses per-SAMPLE statistics (utils_diffusion.py:147-158: std over every axis but
        the batch axis) while the kernel reduces over its whole input, so a batch with guidance rescale is updated sample by sample."""
        f = lambda v: None if v is None else v.float().contiguous()
        x, v_c, v_u = f(x), f(v_c), f(v_u)
        extra = {k: (f(v) if isinstance(v, torch.Tensor) else v) for k, v in extra.items()}
        if x.shape[0] == 1 or v_u is None or sc["guidance_rescale"] <= 0.0:
            return ops.ddim_update(x, v_c, v_u, noise, sc, **extra)
        outs = []
        for b in range(x.shape[0]):
            eb = {k: (v[b:b + 1].contiguous() if isinstance(v, torch.Tensor) else v) for k, v in extra.items()}
            outs.append(ops.ddim_update(x[b:b + 1].contiguous(), v_c[b:b + 1].contiguous(), v_u[b:b + 1].contiguous(), noise[b:b + 1].contiguous(), sc, **eb))
        return torch.cat([o[0] for o in outs], 0), torch.cat([o[1] for o in outs], 0)

    # -- img2img helpers of the reference sampler (ddim.py:288-325) ------------------------------------------------------------
    @torch.no_grad()
    def decode(self, x_latent, cond, t_start, unconditional_guidance_scale=1.0, unconditional_conditioning=None, use_original_steps=False,
               callback=None):
        """The last `t_start` steps of the current schedule starting from `x_latent` (no guidance rescale, like the reference)."""
        if use_original_steps:
            raise NotImplementedError("viewcrafter_b200.DDIMSampler.decode: use_original_steps is not implemented")
        timesteps = self.ddim_timesteps[:t_start]
        total_steps = timesteps.shape[0]
        print(f"Running DDIM Sampling with {total_steps} timesteps")
        x_dec = x_latent
        for i, step in enumerate(np.flip(timesteps)):
            index = total_steps - i - 1
            ts = torch.full((x_latent.shape[0],), int(step), device=x_latent.device, dtype=torch.long)
            x_dec, _ = self.p_sample_ddim(x_dec, cond, ts, index=index, unconditional_guidance_scale=unconditional_guidance_scale,
                                          unconditional_conditioning=unconditional_conditioning, _step=int(step))
            if callback:
                callback(i)
        return x_dec

    @torch.no_grad()
    def stochastic_encode(self, x0, t, use_original_steps=False, noise=None):
        """q(x_t | x_0) with the DDIM tables gathered by INDEX t (ddim.py:310-325): fast, not exactly invertible."""
        if use_original_steps:
            sqrt_ac, sqrt_1mac = self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod
        else:
            sqrt_ac = torch.sqrt(torch.as_tensor(self.ddim_alphas, dtype=torch.float32))
            sqrt_1mac = torch.as_tensor(self.ddim_sqrt_one_minus_alphas, dtype=torch.float32)
        if noise is None:
            noise = torch.randn_like(x0)
        g = lambda a: a.to(x0.device).gather(-1, t.to(x0.device)).reshape(t.shape[0], *((1,) * (x0.dim() - 1)))
        return g(sqrt_ac) * x0 + g(sqrt_1mac) * noise
