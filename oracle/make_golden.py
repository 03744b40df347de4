"""Generate tests/golden/*.npz by running the UNMODIFIED reference (build container only).

    python oracle/make_golden.py            # writes tests/golden/

Every fixture stores inputs, outputs and the (name, shape) list the synthetic weights were
generated from (oracle/synth.py) -- never the weights themselves.  The reference has no tests
or golden vectors of its own (SURVEY.md §4), so these outputs of the reference code are what
pins the oracle.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref_shims, synth  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def _load_synth(module, seed):
    shapes = synth.module_shapes(module)
    module.load_state_dict(synth.synth_state_dict(shapes, seed), strict=True)
    return json.dumps([[n, list(s)] for n, s in shapes])


def gen_schedule():
    ref_shims.install()
    from lvdm.models import utils_diffusion as U
    from lvdm.models.ddpm3d import DDPM
    from lvdm.models.samplers.ddim import DDIMSampler
    out = {}
    for m, S in (("uniform_trailing", 50), ("uniform_trailing", 10), ("uniform_trailing", 3),
                 ("uniform_trailing", 1), ("uniform", 50), ("quad", 20)):
        out[f"ts_{m}_{S}"] = U.make_ddim_timesteps(m, S, 1000, verbose=False)
    out["temb_999_320"] = U.timestep_embedding(torch.tensor([999, 499, 19, 0]), 320).numpy()
    out["temb_10_64"] = U.timestep_embedding(torch.tensor([10]), 64).numpy()
    for base in (0.3, 0.7):
        model = _stub_model(base)
        out[f"alphas_cumprod"] = model.alphas_cumprod.numpy()
        out[f"scale_arr_{base}"] = model.scale_arr.numpy()
        for S, eta in ((50, 1.0), (10, 1.0), (50, 0.0)):
            smp = _cpu_sampler(model)
            smp.make_schedule(S, "uniform_trailing", eta, verbose=False)
            rows = []
            for index in range(S):
                vals = [torch.full((1,), smp.ddim_alphas[index]), torch.full((1,), smp.ddim_alphas_prev[index]),
                        torch.full((1,), smp.ddim_sigmas[index]), torch.full((1,), smp.ddim_sqrt_one_minus_alphas[index]),
                        torch.full((1,), smp.ddim_scale_arr[index]), torch.full((1,), smp.ddim_scale_arr_prev[index])]
                rows.append([v.to(torch.float32).item() for v in vals])
            out[f"step_scalars_b{base}_S{S}_eta{eta}"] = np.asarray(rows, dtype=np.float32)
    np.savez_compressed(os.path.join(OUT, "schedule_kat.npz"), **out)


def _stub_model(base_scale):
    """A bare nn.Module given the reference's own schedule via DDPM.register_schedule (ddpm3d.py:123-186)
    and the scale_arr formula of LatentDiffusion.__init__ (ddpm3d.py:522-527)."""
    ref_shims.install()
    from lvdm.models.ddpm3d import DDPM

    class Stub(torch.nn.Module):
        pass

    m = Stub()
    m.rescale_betas_zero_snr = True
    m.parameterization = "v"
    m.v_posterior = 0.0
    DDPM.register_schedule(m, beta_schedule="linear", timesteps=1000, linear_start=0.00085, linear_end=0.012)
    m.use_dynamic_rescale = True
    m.register_buffer("scale_arr", torch.tensor(np.concatenate((np.linspace(1.0, base_scale, 400), np.full(1000, base_scale))), dtype=torch.float32))
    m.predict_start_from_z_and_v = lambda x, t, v: DDPM.predict_start_from_z_and_v(m, x, t, v)
    m.predict_eps_from_z_and_v = lambda x, t, v: DDPM.predict_eps_from_z_and_v(m, x, t, v)
    m.device = torch.device("cpu")
    return m


def _cpu_sampler(model):
    from lvdm.models.samplers.ddim import DDIMSampler
    smp = DDIMSampler(model)
    smp.register_buffer = lambda name, attr: setattr(smp, name, attr)     # ddim.py:18-22 hard-codes "cuda"
    return smp


def toy_denoiser(x, t, c):
    """Cheap deterministic stand-in for apply_model used by the sampler goldens (both sides call it)."""
    return torch.tanh(0.7 * x * c["k"] + 0.05 * torch.sin(t.float())[:, None, None, None, None]) + 0.1 * c["b"]


def gen_ddim():
    ref_shims.install()
    import lvdm.models.samplers.ddim as ddim_mod
    out = {}
    for tag, S, base in (("S5", 5, 0.3), ("S50", 50, 0.7)):
        model = _stub_model(base)
        model.apply_model = lambda x, t, c, **kw: toy_denoiser(x, t, c)
        g = torch.Generator().manual_seed(11)
        shape = (1, 4, 3, 4, 6)
        x_T = torch.randn(shape, generator=g)
        noises = [torch.randn(shape, generator=g) for _ in range(S)]
        cond = {"b": torch.randn(shape, generator=g), "k": torch.tensor([1.3])}
        uncond = {"b": torch.randn(shape, generator=g), "k": torch.tensor([0.4])}
        it = iter(noises)
        ddim_mod.noise_like = lambda shape_, device, repeat=False: next(it)
        smp = _cpu_sampler(model)
        samples, inter = smp.sample(S=S, batch_size=1, shape=shape[1:], conditioning=cond, eta=1.0, verbose=False,
                                    x_T=x_T, unconditional_guidance_scale=7.5, unconditional_conditioning=uncond,
                                    timestep_spacing="uniform_trailing", guidance_rescale=0.7)
        out[f"{tag}_x_T"] = x_T.numpy(); out[f"{tag}_noises"] = torch.stack(noises).numpy()
        out[f"{tag}_cond_b"] = cond["b"].numpy(); out[f"{tag}_uncond_b"] = uncond["b"].numpy()
        out[f"{tag}_samples"] = samples.numpy()
        out[f"{tag}_n_inter"] = np.asarray(len(inter["x_inter"]))
        out[f"{tag}_pred_x0_last"] = inter["pred_x0"][-1].numpy()
    np.savez_compressed(os.path.join(OUT, "ddim_small.npz"), **out)


def gen_ddim_options():
    """The rarely used switches of the unmodified two-way sampler (ddim.py:136-325) on the toy denoiser: mask / x0 blending (with and
    without clean_cond), a `timesteps` subset, noise_dropout, temperature, precision=16, batch size 2 with guidance rescale (per-sample
    statistics), decode() and stochastic_encode().  Step noise comes from recorded tensors (noise_like is patched); q_sample and
    dropout draw from the global CPU generator after torch.manual_seed -- the product must make the same draws in the same order."""
    ref_shims.install()
    import lvdm.models.samplers.ddim as ddim_mod
    from lvdm.models.ddpm3d import DDPM
    out = {}
    shape = (1, 4, 3, 4, 6)

    def setup(S, seed, base=0.5, shp=shape):
        model = _stub_model(base)
        model.apply_model = lambda x, t, c, **kw: toy_denoiser(x, t, c)
        model.q_sample = lambda x0, t, noise=None: DDPM.q_sample(model, x0, t, noise)
        g = torch.Generator().manual_seed(seed)
        x_T = torch.randn(shp, generator=g)
        noises = [torch.randn(shp, generator=g) for _ in range(S)]
        cond = {"b": torch.randn(shp, generator=g), "k": torch.tensor([1.3])}
        uncond = {"b": torch.randn(shp, generator=g), "k": torch.tensor([0.4])}
        it = iter(noises)
        ddim_mod.noise_like = lambda shape_, device, repeat=False: next(it)
        return model, _cpu_sampler(model), x_T, noises, cond, uncond, g

    def record(tag, x_T, noises, cond, uncond, samples, inter=None):
        out[f"{tag}_x_T"] = x_T.numpy(); out[f"{tag}_noises"] = torch.stack(noises).numpy()
        out[f"{tag}_cond_b"] = cond["b"].numpy(); out[f"{tag}_uncond_b"] = uncond["b"].numpy()
        out[f"{tag}_samples"] = samples.float().numpy()
        if inter is not None:
            out[f"{tag}_n_inter"] = np.asarray(len(inter["x_inter"]))
            out[f"{tag}_pred_x0_last"] = inter["pred_x0"][-1].float().numpy()

    common = dict(batch_size=1, shape=shape[1:], eta=1.0, verbose=False, unconditional_guidance_scale=7.5, timestep_spacing="uniform_trailing",
                  guidance_rescale=0.7)
    for tag, clean in (("mask", False), ("maskclean", True)):
        model, smp, x_T, noises, cond, uncond, g = setup(6, 21)
        x0 = torch.randn(shape, generator=g)
        mask = (torch.rand((1, 1, 3, 4, 6), generator=g) > 0.5).float()
        torch.manual_seed(123)
        samples, inter = smp.sample(S=6, conditioning=cond, x_T=x_T, unconditional_conditioning=uncond, mask=mask, x0=x0,
                                    **(dict(clean_cond=True) if clean else {}), **common)
        record(tag, x_T, noises, cond, uncond, samples, inter)
        out[f"{tag}_x0"] = x0.numpy(); out[f"{tag}_mask"] = mask.numpy()
    # `timesteps` subset: only ddim_sampling takes it (sample() does not forward it)
    model, smp, x_T, noises, cond, uncond, g = setup(10, 22)
    smp.make_schedule(ddim_num_steps=10, ddim_discretize="uniform_trailing", ddim_eta=1.0, verbose=False)
    samples, inter = smp.ddim_sampling(cond, shape, x_T=x_T, timesteps=6, unconditional_guidance_scale=7.5, unconditional_conditioning=uncond,
                                       verbose=False, guidance_rescale=0.7)
    record("subset", x_T, noises, cond, uncond, samples, inter)
    model, smp, x_T, noises, cond, uncond, g = setup(5, 23)
    torch.manual_seed(321)
    samples, inter = smp.sample(S=5, conditioning=cond, x_T=x_T, unconditional_conditioning=uncond, noise_dropout=0.25, **common)
    record("dropout", x_T, noises, cond, uncond, samples, inter)
    model, smp, x_T, noises, cond, uncond, g = setup(5, 24)
    samples, inter = smp.sample(S=5, conditioning=cond, x_T=x_T, unconditional_conditioning=uncond, temperature=0.6, **common)
    record("temp", x_T, noises, cond, uncond, samples, inter)
    model, smp, x_T, noises, cond, uncond, g = setup(5, 25)
    samples, inter = smp.sample(S=5, conditioning=cond, x_T=x_T, unconditional_conditioning=uncond, precision=16, **common)
    record("prec16", x_T, noises, cond, uncond, samples, inter)
    out["prec16_first_inter_dtype"] = np.asarray(str(inter["x_inter"][0].dtype))
    shp2 = (2, 4, 3, 4, 6)
    model, smp, x_T, noises, cond, uncond, g = setup(5, 26, shp=shp2)
    samples, inter = smp.sample(S=5, conditioning=cond, x_T=x_T, unconditional_conditioning=uncond, **dict(common, batch_size=2))
    record("batch2", x_T, noises, cond, uncond, samples, inter)
    # decode(): the last t_start steps of the schedule from a given latent (no guidance rescale, ddim.py:288-308)
    model, smp, x_T, noises, cond, uncond, g = setup(5, 27)
    smp.make_schedule(ddim_num_steps=8, ddim_discretize="uniform_trailing", ddim_eta=1.0, verbose=False)
    x_dec = smp.decode(x_T, cond, 5, unconditional_guidance_scale=7.5, unconditional_conditioning=uncond)
    record("decode", x_T, noises, cond, uncond, x_dec)
    # stochastic_encode(): q(x_t | x_0) with the DDIM alphas gathered by index t (ddim.py:310-325)
    enc_noise = torch.randn(shape, generator=g)
    out["stoch_x0"] = x_T.numpy(); out["stoch_noise"] = enc_noise.numpy()
    out["stoch_out"] = smp.stochastic_encode(x_T, torch.tensor([3]), noise=enc_noise).numpy()
    np.savez_compressed(os.path.join(OUT, "ddim_options.npz"), **out)


def gen_ddim_multicond():
    """The unmodified three-way-CFG sampler (ddim_multiplecond.py) on the toy denoiser: S=5 with cfg_img=2.5 and S=8 with the
    default cfg_img (= the text scale); base 0.3 so that the un-fixed ddim_scale_arr_prev[0] matters."""
    ref_shims.install()
    import lvdm.models.samplers.ddim_multiplecond as mod
    out = {}
    for tag, S, cfg_img in (("S5", 5, 2.5), ("S8", 8, None)):
        model = _stub_model(0.3)
        model.apply_model = lambda x, t, c, **kw: toy_denoiser(x, t, c)
        g = torch.Generator().manual_seed(12)
        shape = (1, 4, 3, 4, 6)
        x_T = torch.randn(shape, generator=g)
        noises = [torch.randn(shape, generator=g) for _ in range(S)]
        cond = {"b": torch.randn(shape, generator=g), "k": torch.tensor([1.3])}
        uncond = {"b": torch.randn(shape, generator=g), "k": torch.tensor([0.4])}
        uncond_img = {"b": torch.randn(shape, generator=g), "k": torch.tensor([0.9])}
        it = iter(noises)
        mod.noise_like = lambda shape_, device, repeat=False: next(it)
        smp = mod.DDIMSampler(model)
        smp.register_buffer = lambda name, attr: setattr(smp, name, attr)
        samples, inter = smp.sample(S=S, batch_size=1, shape=shape[1:], conditioning=cond, eta=1.0, verbose=False,
                                    x_T=x_T, unconditional_guidance_scale=7.5, unconditional_conditioning=uncond,
                                    timestep_spacing="uniform_trailing", guidance_rescale=0.7, cfg_img=cfg_img,
                                    unconditional_conditioning_img_nonetext=uncond_img)
        out[f"{tag}_x_T"] = x_T.numpy(); out[f"{tag}_noises"] = torch.stack(noises).numpy()
        for nm, d in (("cond", cond), ("uncond", uncond), ("uncond_img", uncond_img)):
            out[f"{tag}_{nm}_b"] = d["b"].numpy()
        out[f"{tag}_samples"] = samples.numpy()
        out[f"{tag}_n_inter"] = np.asarray(len(inter["x_inter"]))
        out[f"{tag}_pred_x0_last"] = inter["pred_x0"][-1].numpy()
        out[f"{tag}_scale_prev"] = smp.ddim_scale_arr_prev.numpy()
    np.savez_compressed(os.path.join(OUT, "ddim_multicond_small.npz"), **out)


def gen_unet():
    cases = {
        # name: (unet kwargs overrides, T, H, W)
        "mc64_T4": (dict(model_channels=64), 4, 8, 16),
        "mc64_T16": (dict(model_channels=64), 16, 8, 8),        # 77+16*T == 333 -> per-frame image-token branch
        "mc128_T3": (dict(model_channels=128), 3, 8, 8),
    }
    for name, (over, T, H, W) in cases.items():
        m = ref_shims.build_unet(**over)
        shapes = _load_synth(m, seed=3)
        g = torch.Generator().manual_seed(5)
        x = torch.randn(1, 8, T, H, W, generator=g)
        ctx = torch.randn(1, 333, 1024, generator=g)
        t = torch.tensor([499])
        fs = torch.tensor([10])
        with torch.no_grad():
            y = m(x, t, context=ctx, fs=fs)
        np.savez_compressed(os.path.join(OUT, f"unet_{name}.npz"), shapes=shapes, kwargs=json.dumps(over),
                            x=x.numpy(), ctx=ctx.numpy(), t=t.numpy(), fs=fs.numpy(), y=y.numpy())
        print(name, "out std", float(y.std()), "absmax", float(y.abs().max()))


def gen_vae():
    dec, pq = ref_shims.build_decoder(ch=32)
    shapes_d = _load_synth(dec, seed=4)
    pq.load_state_dict(synth.synth_state_dict(synth.module_shapes(pq), 4))
    g = torch.Generator().manual_seed(6)
    z = torch.randn(2, 4, 8, 12, generator=g)
    with torch.no_grad():
        y = dec(pq(z))
    np.savez_compressed(os.path.join(OUT, "vae_ch32.npz"), shapes=shapes_d, z=z.numpy(), y=y.numpy())
    print("vae out std", float(y.std()))


def gen_vae_enc():
    """Encoder + quant_conv + DiagonalGaussianDistribution.sample of the unmodified reference (autoencoder.py:97-102)."""
    enc, qc = ref_shims.build_encoder(ch=32)
    from lvdm.distributions import DiagonalGaussianDistribution
    shapes_e = _load_synth(enc, seed=14)
    qc.load_state_dict(synth.synth_state_dict(synth.module_shapes(qc), 14))
    g = torch.Generator().manual_seed(16)
    x = torch.rand(2, 3, 32, 48, generator=g) * 2 - 1
    noise = torch.randn(2, 4, 4, 6, generator=g)
    with torch.no_grad():
        moments = qc(enc(x))
        z = DiagonalGaussianDistribution(moments).sample(noise=noise)
    np.savez_compressed(os.path.join(OUT, "vae_enc_ch32.npz"), shapes=shapes_e, x=x.numpy(), moments=moments.numpy(),
                        noise=noise.numpy(), z=z.numpy())
    print("vae enc moments std", float(moments.std()), "z std", float(z.std()))


def gen_resampler():
    """Resampler.forward of the unmodified reference (resampler.py:96-145) at a reduced width; B=2 so the
    latents.repeat batch path is covered.  33 CLIP tokens + 4x4 latents -> 49 keys (ragged vs. the 128-key tile)."""
    over = dict(dim=256, depth=2, dim_head=64, heads=4, num_queries=4, embedding_dim=320, output_dim=192, video_length=4)
    m = ref_shims.build_resampler(**over)
    shapes = _load_synth(m, seed=17)
    g = torch.Generator().manual_seed(18)
    x = torch.randn(2, 33, 320, generator=g)
    with torch.no_grad():
        y = m(x)
    np.savez_compressed(os.path.join(OUT, "resampler_d256.npz"), shapes=shapes, kwargs=json.dumps(over), x=x.numpy(), y=y.numpy())
    print("resampler out std", float(y.std()))


DROPIN_CASES = ((False, 16), (True, 16), (False, 5))     # (multiple_cond_cfg, T)
DROPIN_STRIDE = 17                                       # every 17th output value is stored: ~15k of the 197k at T = 16


def gen_dropin():
    """The reference's own pipeline end to end: its VIPLatentDiffusion from its YAML (configs/inference_pvd_1024.yaml, reduced
    widths, the two OpenCLIP towers replaced by the toys of oracle/synth.py) and its utils.diffusion_utils.image_guided_synthesis
    with its own samplers.  T = 16: 77 + 16 T = 333 context tokens -> per-frame image tokens (openaimodel3d.py:556-560); T = 5: the
    shared-context branch the 25-frame checkpoints take.  Stored: the constructor arguments, the (name, shape) list of the three
    networks' weights (seed 81), the synthesis arguments and a strided sample of each output with the std of the whole output."""
    import yaml
    ref_shims.install()
    import utils.diffusion_utils as DU
    import lvdm.models.samplers.ddim as ref_ddim
    import lvdm.models.samplers.ddim_multiplecond as ref_multi

    def on_cpu(cls):                                      # ddim.py:18-22 hard-codes "cuda"
        return type("CpuSampler", (cls,), {"register_buffer": lambda self, name, attr: setattr(self, name, attr)})

    DU.DDIMSampler, DU.DDIMSampler_multicond = on_cpu(ref_ddim.DDIMSampler), on_cpu(ref_multi.DDIMSampler)
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REF_ROOT, "configs", "inference_pvd_1024.yaml")))["model"]
    P = cfg["params"]
    P["unet_config"]["params"].update(model_channels=64, use_checkpoint=False)
    P["first_stage_config"]["params"]["ddconfig"].update(ch=32)
    P["cond_stage_config"] = {"target": "oracle.synth.ToyText"}
    P["img_cond_stage_config"] = {"target": "oracle.synth.ToyImage"}
    P["image_proj_stage_config"]["params"].update(dim=128, depth=1, heads=2, embedding_dim=64)      # still 16 x 16 queries -> 1024

    class _AD(dict):                                      # OmegaConf's attribute access, as instantiate_from_config reads it
        __getattr__ = dict.__getitem__

    def ad(x):
        return _AD({k: ad(v) for k, v in x.items()}) if isinstance(x, dict) else [ad(v) for v in x] if isinstance(x, list) else x

    torch.manual_seed(0)
    ref = DU.instantiate_from_config(ad(cfg)).eval()
    nets = ("model.", "first_stage_model.", "image_proj_model.")
    shapes = [(k, s) for k, s in synth.module_shapes(ref) if k.startswith(nets)]
    ref.load_state_dict(synth.synth_state_dict(shapes, seed=81), strict=False)
    out = {"shapes": json.dumps([[n, list(s)] for n, s in shapes]),
           "unet_config": json.dumps(P["unet_config"]["params"]),
           "first_stage_config": json.dumps(P["first_stage_config"]["params"]),
           "image_proj_config": json.dumps(P["image_proj_stage_config"]["params"]),
           "model_params": json.dumps({k: v for k, v in P.items() if not isinstance(v, dict)}),
           "stride": np.asarray(DROPIN_STRIDE)}
    H, W = 8, 8
    for multi, T in DROPIN_CASES:
        videos = torch.rand(1, 3, T, 8 * H, 8 * W, generator=torch.Generator().manual_seed(7)) * 2 - 1
        kw = dict(n_samples=1, ddim_steps=(1 if multi else 2), ddim_eta=1.0, unconditional_guidance_scale=7.5, cfg_img=(2.0 if multi else None),
                  fs=10, text_input=True, multiple_cond_cfg=multi, timestep_spacing="uniform_trailing", guidance_rescale=0.7, condition_index=[0])
        torch.manual_seed(11)
        y = DU.image_guided_synthesis(ref, ["a photo"], videos, [1, 4, T, H, W], **kw)
        tag = f"multi{int(multi)}_T{T}"
        out[f"{tag}_kwargs"] = json.dumps(kw)
        out[f"{tag}_shape"] = np.asarray(y.shape)
        out[f"{tag}_std"] = np.asarray(float(y.std()))
        out[f"{tag}_sample"] = y.reshape(-1)[::DROPIN_STRIDE].numpy()
        print(tag, "out std", float(y.std()), "stored", out[f"{tag}_sample"].size)
    np.savez_compressed(os.path.join(OUT, "dropin_pipeline.npz"), **out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["schedule", "ddim", "ddim_options", "ddim_multicond", "unet", "vae", "vae_enc", "resampler", "dropin"]
    with torch.no_grad():
        for w in which:
            globals()["gen_" + w]()
    print("golden fixtures written to", OUT)
