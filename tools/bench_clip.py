"""Whole-clip time of image_guided_synthesis at the flagship size, per stage, with the VAE stages replicated on every rank or split
by frame over the ranks.  Writes one JSON file (--out) on rank 0.

  python tools/bench_clip.py --out DIR/clip_n1.json                                  1 GPU
  python -m torch.distributed.run --nproc-per-node N tools/bench_clip.py --out ...   N GPUs (parallel.shard_model)

Workload: renders 1 x 3 x 25 x 576 x 1024 -> latent 1 x 4 x 25 x 72 x 128, 50-step uniform_trailing DDIM, CFG 7.5, guidance rescale
0.7, eta 1, full-width U-Net (CUDA graph replay) and VAE (per-frame, the shipped default) with synthetic weights, the toy OpenCLIP towers
and reduced Resampler of tools/clip_check.py (the conditioning is not what is measured).  Stages: encode (get_latent_z), decode (per
n_samples variant), denoise = the rest of the call (the sampling loop; the toy conditioning is a few ms).  Each stage is timed with the
host clock between a barrier + device synchronize and a device synchronize, and the slowest rank's time is reported.

Arms, alternating within the call after one untimed clip each (graph capture, weight packing):
  replicated  model._vae detached: every rank encodes and decodes all 25 frames itself (the only arm on one GPU)
  sharded     N > 1: rank r encodes and decodes its frames, the rest is all-gathered (parallel.vae_encode_sharded / vae_decode_sharded)
The max |video difference| between the arms' outputs of the same seed is reported beside the times."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch


def cards():
    """Name and power limit of every GPU of the box (read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return [ln.strip() for ln in r.stdout.splitlines() if ln.strip()]
    except Exception as e:                      # the times are reported either way; the card line says why it is missing
        return [f"{torch.cuda.get_device_name(0)} (power limit not read: {e!r})"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3, help="timed clips per arm")
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_clip.py: no CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from clip_check import clip_model
    from viewcrafter_b200 import parallel, synthesis
    from viewcrafter_b200.configs import UNET_PARAMS

    T, H, W = 25, 72, 128
    model = clip_model(UNET_PARAMS["model_channels"], dev, seed=0)
    comm = None
    if world > 1:
        parallel.shard_model(model, dist, rank, world)
        comm = model._vae
    videos = (torch.rand(1, 3, T, 8 * H, 8 * W, generator=torch.Generator().manual_seed(1)) * 2 - 1).to(dev)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    acc = {"encode": 0.0, "decode": 0.0}
    inside = [False]

    def timed(name, fn):
        def run(*a, **k):
            if inside[0]:                        # vae_decode_sharded calls decode_first_stage: count the outer call only
                return fn(*a, **k)
            inside[0] = True
            sync()
            t0 = time.perf_counter()
            try:
                r = fn(*a, **k)
                torch.cuda.synchronize()
            finally:
                inside[0] = False
            acc[name] += time.perf_counter() - t0
            return r
        return run

    synthesis.get_latent_z = timed("encode", synthesis.get_latent_z)
    parallel.vae_decode_sharded = timed("decode", parallel.vae_decode_sharded)
    model.decode_first_stage = timed("decode", model.decode_first_stage)

    def clip(arm):
        model._vae = comm if arm == "sharded" else None
        acc["encode"] = acc["decode"] = 0.0
        torch.manual_seed(2)
        sync()
        t0 = time.perf_counter()
        out = synthesis.image_guided_synthesis(model, ["a photo"], videos, [1, 4, T, H, W], n_samples=1, ddim_steps=args.steps, ddim_eta=1.0,
                                               unconditional_guidance_scale=7.5, fs=10, text_input=True, timestep_spacing="uniform_trailing",
                                               guidance_rescale=0.7, condition_index=[0])
        torch.cuda.synchronize()
        total = time.perf_counter() - t0
        t = torch.tensor([total, acc["encode"], acc["decode"]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total, enc, dec = (float(v) * 1e3 for v in t)
        return out, dict(total_ms=total, encode_ms=enc, decode_ms=dec, denoise_ms=total - enc - dec)

    arms = ["replicated", "sharded"] if world > 1 else ["replicated"]
    outs = {}
    for arm in arms:
        outs[arm], _ = clip(arm)                 # untimed: graph capture, weight packing, NCCL warm-up
    runs = {arm: [] for arm in arms}
    for _ in range(args.reps):
        for arm in arms:
            outs[arm], r = clip(arm)
            runs[arm].append(r)
    diff = None
    if world > 1:
        d = (outs["replicated"] - outs["sharded"]).abs().max().reshape(1).double()
        dist.all_reduce(d, op=dist.ReduceOp.MAX)
        diff = float(d)
    finite = all(bool(torch.isfinite(o).all()) for o in outs.values())

    if rank == 0:
        def summary(rs):
            s = {}
            for k in rs[0]:
                v = np.array([r[k] for r in rs])
                s[k] = dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()), spread=float((v.max() - v.min()) / np.median(v)))
            return s

        layout = "1 GPU" if world == 1 else ("2-way CFG split x %d-way frame sharding" % (world // 2) if world % 2 == 0 else "%d-way frame sharding" % world)
        res = {"tool": "tools/bench_clip.py", "n_gpus": world, "unet_layout": layout, "cards": cards(),
               "workload": "image_guided_synthesis: renders 1x3x25x576x1024, latent 1x4x25x72x128, %d DDIM steps uniform_trailing, CFG 7.5, "
                           "guidance_rescale 0.7, eta 1, two-way CFG; full-width U-Net (CUDA graph) and VAE (perframe_ae) with synthetic weights; "
                           "toy OpenCLIP towers and reduced Resampler" % args.steps,
               "timing": "host clock between barrier + device synchronize and device synchronize; slowest rank; denoise = total - encode - decode",
               "vae_frames_per_rank": [f1 - f0 for f0, f1 in parallel.frame_ranges(T, world)],
               "reps": args.reps, "arms": {arm: {"runs": rs, "summary": summary(rs)} for arm, rs in runs.items()},
               "max_abs_video_diff_replicated_vs_sharded": diff, "finite": finite}
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({a: {k: round(v["median"], 1) for k, v in r["summary"].items()} for a, r in res["arms"].items()}), "diff", diff, flush=True)
    sys.stdout.flush()
    if world > 1:                                # as bench.py: no process-group teardown after captured collectives
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)


if __name__ == "__main__":
    main()
