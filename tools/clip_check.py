"""torchrun target: the VAE stages of a clip split by frame over the ranks vs one GPU, then a whole image_guided_synthesis under
parallel.shard_model vs one GPU (rank 0 prints, CLIP_CHECK_OK on success).

  1. Full-width VAE (ch=128, synthetic weights of oracle/synth.py), one clip of 25 frames at 576x1024.  Every rank first runs the
     single-GPU get_latent_z and decode_first_stage itself, then the sharded ones (parallel.vae_encode_sharded / vae_decode_sharded),
     and compares what it gathered with what it computed alone: per-frame mode (perframe_ae, the shipped default) must be
     bit-identical, batched mode (a rank runs its N_local frames per call instead of 25) within 0.03 std.
  2. image_guided_synthesis, 3 DDIM steps at 25 x 72 x 128 latents, U-Net at model_channels=64, the ToyText / ToyImage towers of
     oracle/synth.py and a reduced Resampler, CUDA graph on, two-way and three-way CFG: sharded vs single GPU within 0.15 (the
     sharded-step bound of tools/parallel_check.py; the VAE stages add nothing to it in per-frame mode).

VC_PEER_COMM=1 (default) / 0 selects the U-Net's frame exchange (NVLink peer memory / NCCL); the VAE gathers always use NCCL.
--shared-gpu puts every rank on cuda:0 and uses gloo (the gathers go through host memory), so that a box with one GPU runs the sharded
code on the real kernels; only world 2 (CFG split: the U-Net exchanges no frames) is supported that way.
clip_model() is shared with tools/bench_clip.py."""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch


def clip_model(model_channels: int, device, seed: int = 0):
    """LatentDiffusion with the U-Net at `model_channels`, the full-width VAE and the attributes image_guided_synthesis reads:
    ToyText / ToyImage towers, a Resampler at the reduced width of tests/golden/dropin_pipeline.npz, uncond_type "empty_seq".
    Weights: oracle/synth.py from (name, shape, seed)."""
    from oracle import synth
    from viewcrafter_b200.configs import UNET_PARAMS, VAE_DDCONFIG
    from viewcrafter_b200.diffusion import LatentDiffusion
    from viewcrafter_b200.resampler import Resampler

    class Model(LatentDiffusion):
        def __init__(self):
            super().__init__(dict(UNET_PARAMS, model_channels=model_channels), dict(ddconfig=VAE_DDCONFIG, embed_dim=4), base_scale=0.3)
            self.uncond_type = "empty_seq"
            self.cond_stage_model = synth.ToyText()
            self.embedder = synth.ToyImage()
            self.image_proj_model = Resampler(dim=128, depth=1, dim_head=64, heads=2, num_queries=16, embedding_dim=64, output_dim=1024,
                                              ff_mult=4, video_length=16)

        def get_learned_conditioning(self, c):
            return self.cond_stage_model.encode(c)

    torch.manual_seed(seed)
    m = Model()
    sd = m.state_dict()
    sd.update(synth.synth_state_dict([(k, s) for k, s in synth.module_shapes(m) if k.startswith(("model.", "first_stage_model.", "image_proj_model."))],
                                     seed=seed))
    m.load_state_dict(sd, strict=True)
    return m.to(device).eval()


def main():
    import torch.distributed as dist
    ap = argparse.ArgumentParser()
    ap.add_argument("--shared-gpu", action="store_true", help="every rank on cuda:0, gloo process group (world 2 only)")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    if args.shared_gpu:
        assert world == 2, "--shared-gpu: only the CFG split of world 2 runs without a frame exchange in the U-Net"
        local = 0
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.shared_gpu:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=dev)
    from viewcrafter_b200 import parallel
    from viewcrafter_b200.synthesis import get_latent_z, image_guided_synthesis

    T, H, W = 25, 72, 128
    model = clip_model(64, dev, seed=5)
    g = torch.Generator().manual_seed(6)
    videos = (torch.rand(1, 3, T, 8 * H, 8 * W, generator=g) * 2 - 1).to(dev)
    latents = torch.randn(1, 4, T, H, W, generator=g).to(dev)

    def timed(fn, *a):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        r = fn(*a)
        torch.cuda.synchronize()
        return r, (time.perf_counter() - t0) * 1e3

    def vae_stages(sharded):
        out = {}
        for pf in (True, False):
            model.perframe_ae = pf
            torch.manual_seed(7)
            z, t_enc = timed(get_latent_z, model, videos)
            state = torch.get_rng_state()
            y, t_dec = timed(lambda: parallel.vae_decode_sharded(model, latents) if sharded else model.decode_first_stage(latents))
            out[pf] = (z, y, state, t_enc, t_dec)
        model.perframe_ae = True
        return out

    kw = dict(n_samples=1, ddim_steps=3, ddim_eta=1.0, unconditional_guidance_scale=7.5, fs=10, text_input=True,
              timestep_spacing="uniform_trailing", guidance_rescale=0.7, condition_index=[0])

    def clips():
        res = {}
        for multi in (False, True):
            torch.manual_seed(11)
            res[multi] = image_guided_synthesis(model, ["a photo"], videos, [1, 4, T, H, W], multiple_cond_cfg=multi,
                                                cfg_img=7.5 if multi else None, **kw)
        return res

    with torch.no_grad():
        single_vae = vae_stages(False)
        single_clip = clips()
        comm = parallel.shard_model(model, dist, rank, world)
        assert model._vae is not None and model._vae.world == world
        sharded_vae = vae_stages(True)
        sharded_clip = clips()

    ok = True
    lines = []
    for pf in (True, False):
        z1, y1, s1, te1, td1 = single_vae[pf]
        z2, y2, s2, te2, td2 = sharded_vae[pf]
        ez, ey = float((z1 - z2).abs().max()), float((y1 - y2).abs().max())
        same = torch.equal(z1, z2) and torch.equal(y1, y2)
        good = torch.equal(s1, s2) and (same if pf else (ez <= 0.03 * float(z1.std()) and ey <= 0.03 * float(y1.std())))
        ok = ok and good
        lines.append(f"[rank {rank}] VAE {'per-frame' if pf else 'batched'}: sharded == single-GPU bit for bit: {same}; max |latent diff| {ez:.3g} "
                     f"(std {float(z1.std()):.3g}), max |video diff| {ey:.3g} (std {float(y1.std()):.3g}); RNG state equal {torch.equal(s1, s2)}; "
                     f"encode {te1:.1f} -> {te2:.1f} ms, decode {td1:.1f} -> {td2:.1f} ms")
    d = torch.tensor([float((sharded_clip[m] - single_clip[m]).abs().max()) for m in (False, True)], device=dev)
    dist.all_reduce(d, op=dist.ReduceOp.MAX)
    finite = all(bool(torch.isfinite(v).all()) for v in sharded_clip.values())
    ok = ok and finite and float(d.max()) < 0.15 and all(sharded_clip[m].shape == (1, 1, 3, T, 8 * H, 8 * W) for m in (False, True))
    for ln in lines:
        print(ln, flush=True)
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = bool(flag.item() > 0)
    if rank == 0:
        layout = f"CFG split 2 x {world // 2} frames" if getattr(model, "_cfg", None) is not None else f"{world}-way frames"
        where = "all ranks on one GPU, gloo" if args.shared_gpu else "NCCL"
        print(f"world {world} ({layout}, {where}, U-Net comm {type(comm).__name__ if comm else 'none'}): image_guided_synthesis 3 steps "
              f"|sharded - single| two-way {float(d[0]):.4g}, three-way {float(d[1]):.4g} (video std {float(single_clip[False].std()):.3g})", flush=True)
        if ok:
            print("CLIP_CHECK_OK", flush=True)
    # leave like bench.py does: no process-group teardown after NCCL collectives were captured into CUDA graphs
    sys.stdout.flush(); sys.stderr.flush()
    torch.cuda.synchronize()
    dist.barrier()
    os._exit(0 if ok else 1)


if __name__ == "__main__":
    main()
