"""Three-way (text + image) guidance throughput: DDIM steps/s of ddim_multiplecond.DDIMSampler at the flagship size (latent
1x4x25x72x128, CFG 7.5, cfg_img 7.5, guidance_rescale 0.7, eta 1, 50-step uniform_trailing schedule, the U-Net replayed as a CUDA
graph unless --no-graph).  Prints the card name and power limit and one JSON line per arm.

  python tools/bench_multicond.py                       1 GPU: alternates, in one process,
        "b2+b1"   the previous three-way step: a B=2 (cond, uncond) forward with the shared prefix + a B=1 image-only forward
        "b3"      the batched step: ONE B=3 forward with the prefix computed once
        "twoway"  the two-way step of ddim.DDIMSampler (B=2 forward) for reference
      and compares b2+b1 and b3 outputs of the same step from the same latent and noise seed.
  torchrun --nproc-per-node N tools/bench_multicond.py  N GPUs (parallel.shard_model; CFG split unless --no-cfg-split): the b3 step
      and the two-way step only (the previous three-way step did not run on the split layout)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info(index):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:                      # the numbers are reported either way; the card line says why it is missing
        return f"{torch.cuda.get_device_name(index)} (power limit not read: {e!r})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=6, help="timed steps per arm and round")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm before the first round (include the graph capture)")
    ap.add_argument("--rounds", type=int, default=2, help="the arms alternate this many times")
    ap.add_argument("--workload", default="ViewCrafter_25")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cfg-split", action="store_true")
    args = ap.parse_args()
    import bench
    from viewcrafter_b200.ddim import DDIMSampler as TwoWay
    from viewcrafter_b200.ddim_multiplecond import DDIMSampler as ThreeWay

    class PreviousThreeWay(ThreeWay):
        """The three-way step before the batched B=3 forward: _apply_both (B=2 with the shared prefix) + a separate B=1 forward."""

        def _apply_three(self, x, t, c, uc, uc_img, kwargs):
            v_c, v_u = self._apply_both(x, t, c, uc, kwargs)
            return v_c, v_u, self.model.apply_model(x, t, uc_img, **kwargs)

    wl = bench.WORKLOADS[args.workload]
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_multicond.py: no CUDA device")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    model = bench.build_model(wl, device)
    if world > 1:
        from viewcrafter_b200 import parallel
        parallel.shard_model(model, dist, rank, world, cfg_split=not args.no_cfg_split)
    if not args.no_graph:
        model.model.diffusion_model.enable_cuda_graph()
    _, dev = bench.synthetic_inputs(wl, device)
    c, uc = bench.conds(dev, None)
    ctx_i = torch.randn(1, 333, 1024, generator=torch.Generator().manual_seed(3)).to(device)
    uc_img = {"c_crossattn": [ctx_i], "c_concat": [dev["c_concat"]]}
    fs = torch.tensor([10], device=device, dtype=torch.long)
    arms = {"b3": ThreeWay(model, batch_cfg=True), "twoway": TwoWay(model, batch_cfg=True)}
    if world == 1:
        arms = {"b2+b1": PreviousThreeWay(model, batch_cfg=True), **arms}
    for s in arms.values():
        s.make_schedule(50, "uniform_trailing", 1.0, verbose=False)
    order = np.flip(arms["b3"].ddim_timesteps)

    def step(name, x, i):
        i %= 50
        ts = torch.full((1,), int(order[i]), device=device, dtype=torch.long)
        kw = dict(index=50 - i - 1, unconditional_guidance_scale=7.5, unconditional_conditioning=uc, fs=fs, guidance_rescale=0.7, _step=int(order[i]))
        if name != "twoway":
            kw.update(cfg_img=7.5, unconditional_conditioning_img_nonetext=uc_img)
        return arms[name].p_sample_ddim(x, c, ts, **kw)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # same step, same latent, same noise draw: the outputs of the previous and the batched three-way step
    outs = {}
    for name in arms:
        if name != "twoway":
            torch.manual_seed(11)
            outs[name] = step(name, dev["x_T"], 10)[0].float()
    diff = float((outs["b2+b1"] - outs["b3"]).abs().max()) if "b2+b1" in outs else None
    for name in arms:
        x = dev["x_T"]
        for i in range(args.warmup):
            x, _ = step(name, x, i)
    sync()
    times = {name: [] for name in arms}
    for _ in range(args.rounds):
        for name in arms:
            x = dev["x_T"]
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                x, _ = step(name, x, args.warmup + i)
            e1.record()
            sync()
            times[name].append(e0.elapsed_time(e1) / args.steps)
    if rank == 0:
        print(f"card: {card_info(local)}; {world} GPU(s)", flush=True)
        layout = "1 GPU" if world == 1 else ("CFG split 2 x %d frames" % (world // 2) if (world % 2 == 0 and not args.no_cfg_split) else "%d-way frames" % world)
        for name, ms in times.items():
            line = {"arm": name, "layout": layout, "steps_per_s": 1e3 / float(np.median(ms)), "ms_per_step_rounds": [round(v, 2) for v in ms],
                    "workload": "%s latent 1x4x%dx%dx%d, CFG 7.5, cfg_img 7.5" % (args.workload, wl["T"], wl["H"], wl["W"]),
                    "graph": not args.no_graph, "steps": args.steps, "rounds": args.rounds}
            if name == "b3" and diff is not None:
                line["max_abs_diff_vs_b2+b1"] = diff
            print(json.dumps(line), flush=True)
    sys.stdout.flush()
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)                     # as bench.py: no process-group teardown after captured collectives


if __name__ == "__main__":
    main()
