#!/usr/bin/env python
"""bench.py -- DDIM denoise-steps/sec of the ViewCrafter hot path on B200 (contract: task brief, BASELINE.json).

    python bench.py --gpus 1 --steps 4 --warmup 3                 # our arm, headline workload 25x4x72x128
    python bench.py --impl reference --steps 2 --warmup 1         # the reference's algorithm on the host CPU cores
    python bench.py --steps 4 --warmup 3 --dump-outputs DIR       # + the last timed step's x_prev / pred_x0 as DIR/*.npy
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # frame/CFG-sharded, N in {2,4,8}

One "step" = one DDIMSampler.p_sample_ddim: 2 U-Net forwards (cond + uncond, CFG 7.5), guidance rescale 0.7,
v-prediction update with eta=1 noise.  Data is synthetic (random-init weights of the shipped architecture with the
zero-initialised tensors re-drawn, random latents / render-latents / context), as BASELINE.md config 3 specifies.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "ViewCrafter_25": dict(T=25, H=72, W=128, base_scale=0.3, px="576x1024"),
    "ViewCrafter_25_512": dict(T=25, H=40, W=64, base_scale=0.7, px="320x512"),
    "ViewCrafter_16": dict(T=16, H=72, W=128, base_scale=0.3, px="576x1024"),
}
UNET_FWD_TFLOP = {"ViewCrafter_25": 82.76, "ViewCrafter_25_512": 20.19, "ViewCrafter_16": 52.34}   # SURVEY.md 8(d) / BASELINE.md 2
A100_README_STEPS_PER_S = {"ViewCrafter_25": 50 / 120.0, "ViewCrafter_25_512": 50 / 50.0, "ViewCrafter_16": 50 / 75.0}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
def build_model(wl, device):
    from viewcrafter_b200.configs import UNET_PARAMS
    from viewcrafter_b200.diffusion import LatentDiffusion
    torch.manual_seed(0)
    with torch.device(device):
        model = LatentDiffusion(UNET_PARAMS, None, base_scale=wl["base_scale"])
    g = torch.Generator(device=device).manual_seed(1)
    with torch.no_grad():
        for p in model.parameters():                       # zero-init layers would make the network output exactly 0
            if float(p.detach().abs().max()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g, device=device) * 0.02)
    return model.eval()


def synthetic_inputs(wl, device, pinned=False):
    g = torch.Generator().manual_seed(2)
    T, H, W = wl["T"], wl["H"], wl["W"]
    mk = lambda *s: torch.randn(*s, generator=g)
    host = dict(x_T=mk(1, 4, T, H, W), c_concat=mk(1, 4, T, H, W), ctx_c=mk(1, 333, 1024), ctx_u=mk(1, 333, 1024))
    if pinned:
        host = {k: v.pin_memory() for k, v in host.items()}
    dev = {k: v.to(device) for k, v in host.items()}
    return host, dev


def conds(d, fs):
    c = {"c_crossattn": [d["ctx_c"]], "c_concat": [d["c_concat"]]}
    uc = {"c_crossattn": [d["ctx_u"]], "c_concat": [d["c_concat"]]}
    return c, uc


def time_kernel(fn, reps=5):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def kernel_rooflines(wl, device, peaks):
    """Dominant kernels timed alone with CUDA events on the launching (current) stream; operands exceed L2 (126 MB)."""
    from viewcrafter_b200 import ops
    T, H, W = wl["T"], wl["H"], wl["W"]
    M, C = T * H * W, 320
    x = torch.randn(M, C, device=device).half()
    w9 = (torch.randn(9 * C, C, device=device) * 0.02).half()
    t_conv = time_kernel(lambda: ops.conv3x3(x, T, H, W, w9))
    fl_conv = 2.0 * M * 9 * C * C
    heads = 5
    qkv = torch.randn(M, 3 * C, device=device).half()
    t_att = time_kernel(lambda: ops.flash_attn(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], T, H * W, H * W, heads))
    fl_att = 4.0 * T * heads * (H * W) ** 2 * 64
    gam, bet = torch.ones(C, device=device), torch.zeros(C, device=device)
    # the shipped GroupNorm path for this tensor: the producing conv's epilogue leaves the partial sums (gn_out), GroupNorm = finalize + ONE pass
    y = ops.conv3x3(x, T, H, W, w9, gn_out=True)
    gn_parts = ops.gn_part_of(y) is not None
    n_gn0 = ops.gn_from_parts_calls
    t_gn = time_kernel(lambda: ops.groupnorm(y, T, gam, bet, 1e-5, True))
    gn_parts = gn_parts and ops.gn_from_parts_calls > n_gn0
    by_gn = 2.0 * M * C * 2                                     # algorithmic: read once + write once, fp16
    r = {
        "roofline": {"kernel": "gemm_tap2_kernel<160> (tcgen05 cta_group::2 tap-GEMM, 3x3 conv 320->320 @%dx%dx%d)" % (T, H, W), "bound": "tensor",
                     "achieved": fl_conv / t_conv / 1e12, "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
                     "frac": fl_conv / t_conv / 1e12 / peaks["tflops_burst"], "traffic": None, "ms": t_conv * 1e3,
                     "peak_source": peaks["src"] + " cuBLAS bf16 burst", "algorithmic_flop": fl_conv,
                     "algorithmic_bytes": 2.0 * M * C * 2 + 9 * C * C * 2},
        "roofline_attention": {"kernel": "flash_attn_d64_kernel (spatial self-attn, %d heads, N=%d)" % (heads, H * W), "bound": "tensor",
                               "achieved": fl_att / t_att / 1e12, "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
                               "frac": fl_att / t_att / 1e12 / peaks["tflops_burst"], "traffic": None, "ms": t_att * 1e3,
                               "algorithmic_flop": fl_att, "algorithmic_bytes": 4.0 * M * C * 2},
        "roofline_groupnorm": {"kernel": ("gn_part_finalize_kernel + gn_apply_kernel (GroupNorm32+SiLU, C=320; statistics from the producing conv's epilogue, one pass)"
                                          if gn_parts else "gn_fused_kernel (GroupNorm32+SiLU, C=320, statistics pass + normalise pass in one launch)"), "bound": "hbm",
                               "achieved": by_gn / t_gn / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                               "frac": by_gn / t_gn / 1e9 / peaks["hbm_gbs"], "traffic": None, "ms": t_gn * 1e3, "algorithmic_bytes": by_gn},
    }
    # measured DRAM traffic per launch of the same kernels/shapes, from the committed ncu --set full capture (not re-measured
    # here: a number taken under a profiler is never a bench value, and ncu cannot run inside the timed process)
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r0*_ncu_traffic.json")))
    tp = cands[-1] if cands else ""                                       # the newest committed capture
    if tp and (T, H, W) == (25, 72, 128):                                  # the capture is of the headline shapes only
        t = json.load(open(tp))
        if not gn_parts and "groupnorm_fused_statistics_pass" in t:
            t["roofline_groupnorm"] = t["groupnorm_fused_statistics_pass"]
        for k in r:
            if k in t:
                r[k]["traffic"] = t[k]["traffic_bytes"]
                r[k]["traffic_source"] = t["source"].split(" (")[0] + "; " + t[k]["note"]
    return r


def _cpu_threads():
    """Host threads for the CPU legs: the GPU box reports 128 logical CPUs, but the oracle's many mid-sized fp32 ops stop
    scaling (and at 128 threads collapse) well before that; 32 is the plateau of the large U-Net GEMMs."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cores = max(1, min(avail, int(os.environ.get("VC_BENCH_CPU_THREADS", "32"))))
    torch.set_num_threads(cores)
    return cores


def cpu_frame_sample(wl, sd_cpu, steps, warmup, workload_name):
    """The reference's algorithm (oracle port, fp32 torch-CPU) on a BOUNDED sample of the workload: ONE U-Net forward of ONE of
    the T frames at the workload's own latent resolution (every GEMM / conv / attention has its real per-frame shape: e.g.
    9216 x 9216 attention per head at 72x128).  All spatial ops are independent per frame and the temporal ops are linear
    in T (their T x T attention core is < 0.3 % of the FLOPs), and a step is two U-Net forwards of identical shape, so
    steps/s of the full workload = 1 / (2 * T * sample seconds).  That factor is an ESTIMATE, stated as such in the line."""
    from oracle import lvdm_oracle as O
    cores = _cpu_threads()
    T, H, W = wl["T"], wl["H"], wl["W"]
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, 8, 1, H, W, generator=g)
    ctx = torch.randn(1, 333, 1024, generator=g)
    fs = torch.tensor([10])

    def one(i):
        ts = torch.full((1,), 999 - 20 * (i % 50), dtype=torch.long)
        with torch.no_grad():
            return O.unet_forward(sd_cpu, x, ts, ctx, fs)

    for i in range(warmup):
        one(i)
    t0 = time.time()
    for i in range(steps):
        one(warmup + i)
    dt = (time.time() - t0) / max(steps, 1)
    value = 1.0 / (2 * T * dt)
    sample = ("%d timed samples after %d warm-up; one sample = ONE fp32 U-Net forward (full-width weights) of ONE frame of the %s workload "
              "at its real latent resolution 1x%dx%d (%.1f s each on %d threads); steps/s = 1/(2 forwards x %d frames x sample s): an "
              "ESTIMATE by frame count, not a measured full step" % (steps, warmup, workload_name, H, W, dt, cores, T))
    return value, dt, cores, sample


def cpu_config1_measured(sd_cpu):
    """BASELINE.json config 1 measured, not scaled: one fp32 U-Net forward of the reference algorithm at the real
    ViewCrafter_25_512 latent 1x8x25x40x64 on the host cores; a CFG DDIM step is two such forwards + a 1 MB update."""
    from oracle import lvdm_oracle as O
    cores = _cpu_threads()
    g = torch.Generator().manual_seed(4)
    x = torch.randn(1, 8, 25, 40, 64, generator=g)
    ctx = torch.randn(1, 333, 1024, generator=g)
    t0 = time.time()
    with torch.no_grad():
        O.unet_forward(sd_cpu, x, torch.tensor([999]), ctx, torch.tensor([10]))
    dt = time.time() - t0
    return {"value": 1.0 / (2 * dt), "unit": "steps/s", "cores": cores, "kind": "port", "forward_s": dt,
            "sample": "BASELINE config 1 at its real size: ONE measured fp32 U-Net forward at latent 25x4x40x64 (%.1f s on %d threads); "
                      "a CFG step = 2 identical forwards (S=1 => %.1f s per step); no FLOP scaling" % (dt, cores, 2 * dt)}


# --------------------------------------------------------------------------------------------------
def gpu_parity_and_eager_baseline(wl, model, dev, sampler, run_step):
    """(1) parity at the bench workload: one U-Net forward (t = 499) of the CUDA path vs the oracle in fp32 on this GPU, with
    E_ref = |oracle under fp16 autocast - oracle fp32| beside it (SURVEY.md 8d tolerance rule: accept <= 2 E_ref);
    (2) the same-box GPU baseline: the reference ALGORITHM in PyTorch eager on this B200 -- the oracle port under
    torch.autocast(fp16) (viewcrafter.py:98) with fused SDPA attention (the reference's xformers path, attention.py:146-190) --
    timed for whole CFG DDIM steps (2 forwards + update) with CUDA events.  /root/reference itself cannot travel to the box."""
    from oracle import lvdm_oracle as O
    unet = model.model.diffusion_model
    sd = {k: v.detach() for k, v in unet.state_dict().items()}
    x, cc, ctx_c, ctx_u = dev["x_T"], dev["c_concat"], dev["ctx_c"], dev["ctx_u"]
    fs = torch.tensor([10], device=x.device, dtype=torch.long)
    xc = torch.cat([x, cc], 1)
    ts = torch.full((1,), 499, device=x.device, dtype=torch.long)
    with torch.no_grad(), O.exact_fp32():
        ref32 = O.unet_forward(sd, xc, ts, ctx_c, fs)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        ref16 = O.unet_forward(sd, xc, ts, ctx_c, fs).float()
    y = unet(xc, ts, context=ctx_c, fs=fs).float()
    err, e_ref = (y - ref32).abs(), (ref16 - ref32).abs()
    parity = {"what": "one U-Net forward at the bench workload (t=499), CUDA path vs the fp32 oracle on the same GPU (TF32 off)",
              "max_abs_err": float(err.max()), "mean_abs_err": float(err.mean()), "e_ref_max": float(e_ref.max()),
              "e_ref_mean": float(e_ref.mean()), "out_std": float(ref32.std()),
              "rule": "accept max <= 2*e_ref_max and mean <= 2*e_ref_mean (e_ref = fp16-autocast oracle vs fp32 oracle)",
              "ok": bool(float(err.max()) <= 2 * float(e_ref.max()) and float(err.mean()) <= 2 * float(e_ref.mean()))}
    del ref32, ref16, y, err, e_ref
    sched = {k: v.to(x.device) for k, v in O.model_schedule(base_scale=wl["base_scale"]).items()}
    tab = O.ddim_tables(sched, 50, "uniform_trailing", 1.0)

    def eager_step(xx, i):
        index = 49 - (i % 50)
        step = int(tab["timesteps"][index])
        tt = torch.full((1,), step, device=x.device, dtype=torch.long)
        xin = torch.cat([xx, cc], 1)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16), O.attention_mode("sdpa"):
            v_c = O.unet_forward(sd, xin, tt, ctx_c, fs).float()
            v_u = O.unet_forward(sd, xin, tt, ctx_u, fs).float()
        noise = torch.randn(xx.shape, device=xx.device)
        return O.ddim_update(xx, v_c, v_u, O.step_scalars(tab, index), sched["sqrt_alphas_cumprod"][step].item(),
                             sched["sqrt_one_minus_alphas_cumprod"][step].item(), noise, 7.5, 0.7)[0]

    xx = eager_step(x, 0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 3
    e0.record()
    for i in range(n):
        xx = eager_step(xx, 1 + i)
    e1.record(); torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3 / n
    eager = {"value": 1.0 / dt, "unit": "steps/s", "ms_per_step": dt * 1e3, "steps": n, "warmup": 1,
             "kind": "oracle port of the reference algorithm in PyTorch eager on this GPU: torch.autocast(fp16), cuDNN/cuBLAS convs and "
                     "linears, F.scaled_dot_product_attention for every attention, two sequential U-Net forwards per step",
             "finite": bool(torch.isfinite(xx).all())}
    return parity, eager


def vae_decode_bench(wl, device):
    """BASELINE config 5: VAE decode frames/s at the workload's frame size, per frame (the reference's perframe_ae loop,
    ddpm3d.py:646-671) and batched (5 frames per call); random-init full-width decoder."""
    from viewcrafter_b200.autoencoder import AutoencoderKL
    from viewcrafter_b200.configs import VAE_DDCONFIG
    torch.manual_seed(0)
    with torch.device(device):
        vae = AutoencoderKL(VAE_DDCONFIG, None, 4).eval()
    n = 5
    z = torch.randn(n, 4, wl["H"], wl["W"], device=device)
    with torch.no_grad():
        t1 = time_kernel(lambda: [vae.decode(z[i:i + 1]) for i in range(n)], reps=2)
        tb = time_kernel(lambda: vae.decode(z), reps=2)
    return {"unit": "frames/s", "per_frame": n / t1, "batched_5": n / tb, "frame": "%dx%d" % (8 * wl["H"], 8 * wl["W"]),
            "tflop_per_frame": 5.754 * wl["H"] * wl["W"] / (72 * 128)}


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ViewCrafter_25", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the parity block and the eager-PyTorch GPU baseline")
    ap.add_argument("--no-vae", action="store_true")
    ap.add_argument("--no-batch-cfg", action="store_true")
    ap.add_argument("--no-cfg-split", action="store_true", help="N > 1: pure frame sharding (every rank runs the B=2 cond+uncond forward on its frames) instead of 2-way CFG split x N/2-way frames")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying the captured forward")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step returned (x_prev, pred_x0) "
                                                          "as DIR/<name>.npy in float32; the same arguments give the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    metric = "DDIM denoise-steps/sec @ %sx%df" % (wl["px"], wl["T"])
    config = {"workload": "%s: latent 1x4x%dx%dx%d, CFG 7.5 (2 U-Net forwards/step), guidance_rescale 0.7, eta 1.0, 50-step uniform_trailing schedule"
                          % (args.workload, wl["T"], wl["H"], wl["W"]),
              "l2": "working set per forward (tens of GB of activations, 2.9 GB weights) exceeds the 126 MB L2; no flush needed",
              "cfg": ("N=1: cond+uncond as one B=2 forward; the context-free prefix (input_blocks.0, init_attn, input_blocks.1 up to "
                      "attn1; 6.9 of 165.5 TFLOP) is computed once for both branches and the cross-attention K/V of the step-invariant "
                      "context are projected once per context tensor -- same outputs as two full forwards (SURVEY.md App. C.1/C.2); "
                      "N>=2 even: one CFG branch per half of the ranks")}

    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import synth
        from viewcrafter_b200.configs import UNET_PARAMS
        from viewcrafter_b200.unet import UNetModel
        with torch.device("meta"):
            shapes = [(k, tuple(v.shape)) for k, v in UNetModel(**UNET_PARAMS).state_dict().items()]
        sd = synth.synth_state_dict(shapes, seed=0)
        # the CPU needs no warm-up beyond the first call (page-in of 5.8 GB of weights): run min(W, 1) untimed samples
        value, dt, cores, sample = cpu_frame_sample(wl, sd, args.steps, min(args.warmup, 1), args.workload)
        line = {"impl": "reference", "metric": metric, "value": value, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config, "estimated": True, "sample_seconds": dt,
                "sample_to_step_factor": 2 * wl["T"],
                "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    from viewcrafter_b200 import _lib
    from viewcrafter_b200.ddim import DDIMSampler
    lib = _lib.load()
    peaks = measured_peaks()

    model = build_model(wl, device)
    if world > 1:
        from viewcrafter_b200 import parallel
        parallel.shard_model(model, dist, rank, world, cfg_split=not args.no_cfg_split)
    if not args.no_graph:
        model.model.diffusion_model.enable_cuda_graph()
    config["host"] = ("eager launches" if args.no_graph else
                      "the U-Net forward is captured once (2nd step) and replayed as one CUDA graph; the warm-up steps include the capture")
    sampler = DDIMSampler(model, batch_cfg=not args.no_batch_cfg)
    sampler.make_schedule(50, "uniform_trailing", 1.0, verbose=False)
    host, dev = synthetic_inputs(wl, device, pinned=True)
    c, uc = conds(dev, None)
    fs = torch.tensor([10], device=device, dtype=torch.long)
    order = np.flip(sampler.ddim_timesteps)

    def run_step(x, i, cc=c, uu=uc):
        i = i % 50
        index = 50 - i - 1
        ts = torch.full((1,), int(order[i]), device=device, dtype=torch.long)
        return sampler.p_sample_ddim(x, cc, ts, index=index, unconditional_guidance_scale=7.5, unconditional_conditioning=uu,
                                     fs=fs, guidance_rescale=0.7, _step=int(order[i]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- N > 1: numerics of the sharded forward against the unsharded one on the same GPU (one forward, t = 499) ----
    unet_m = model.model.diffusion_model
    comm = unet_m._comm
    shard_err = None
    if world > 1 and comm is not None:
        gm = unet_m._graph_mode
        unet_m.enable_cuda_graph(False)
        xc = torch.cat([dev["x_T"], dev["c_concat"]], 1)
        t499 = torch.full((1,), 499, device=device, dtype=torch.long)
        comm.bytes_moved = 0
        if hasattr(comm, "fused_switches"):
            comm.fused_switches = 0
        y_sh = unet_m(xc, t499, context=dev["ctx_c"], fs=fs)
        comm.bytes_per_forward = comm.bytes_moved
        comm.fused_per_forward = getattr(comm, "fused_switches", 0)
        # exposed communication: the exchanges run in-stream, so their device time (transfer + waiting for the slowest peer) is not
        # overlapped with compute; measured over one more eager forward with CUDA events around every exchange / statistics call
        torch.cuda.synchronize(); dist.barrier()
        comm.profile(True)
        fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fe0.record()
        unet_m(xc, t499, context=dev["ctx_c"], fs=fs)
        fe1.record()
        comm.exposed_ms = comm.profile_ms()
        comm.forward_ms = fe0.elapsed_time(fe1)
        comm.n_exchanges = len(comm._prof)
        comm.profile(False)
        unet_m._comm = None
        y_1 = unet_m(xc, t499, context=dev["ctx_c"], fs=fs)
        unet_m._comm = comm
        e = (y_sh - y_1).abs().max().reshape(1)
        dist.all_reduce(e, op=dist.ReduceOp.MAX)
        shard_err = {"max_abs_err": float(e), "out_std": float(y_1.std()),
                     "what": "one U-Net forward (t=499): frame-sharded over this rank's group vs the same weights unsharded on one GPU"}
        del y_sh, y_1
        comm.bytes_moved = 0
        unet_m.enable_cuda_graph(gm)

    # ---- device-resident throughput ("value") ----
    x = dev["x_T"]
    for i in range(args.warmup):
        x, _ = run_step(x, i)
    barrier()
    lib.vc_reset_launch_count()
    unet_m.graph_replayed_launches = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        e0.record()
        for i in range(args.steps):
            x, pred_x0 = run_step(x, args.warmup + i)
        e1.record()
        barrier()
    launches = int(lib.vc_launch_count()) + int(unet_m.graph_replayed_launches)   # host-launched + executed through graph replays
    t_dev = torch.tensor([e0.elapsed_time(e1) * 1e-3], device=device, dtype=torch.float64)
    finite = bool(torch.isfinite(x).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x_prev=x, pred_x0=pred_x0)

    # ---- end to end through the sampler API with HOST buffers: H2D of the step inputs + D2H of x_{t-1} every step ----
    # The sampler API takes the conditioning once per clip (ddim.py:61-134 / utils/diffusion_utils.py:117-201), so it stays
    # resident; what changes every step is the latent: x_t comes from pinned host memory and x_{t-1} goes back to it.
    out_host = torch.empty_like(host["x_T"]).pin_memory()
    x_host = host["x_T"]
    h2d = host["x_T"].numel() * 4
    d2h = out_host.numel() * 4
    config["e2e"] = "per step: H2D x_t from pinned host memory, p_sample_ddim, D2H x_{t-1} + stream sync; conditioning uploaded once per clip"

    def e2e_step(i):
        xd = x_host.to(device, non_blocking=True)
        xn, _ = run_step(xd, i)
        out_host.copy_(xn, non_blocking=True)
        torch.cuda.current_stream().synchronize()             # the caller reads the result
        return out_host

    for i in range(min(args.warmup, 2)):
        e2e_step(i)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(args.steps):
        e2e_step(args.warmup + i)
    f1.record()
    barrier()
    t_e2e = torch.tensor([f0.elapsed_time(f1) * 1e-3], device=device, dtype=torch.float64)
    comm_info = None
    if world > 1:
        from viewcrafter_b200 import parallel as _par
        cfg_split = world % 2 == 0 and not args.no_cfg_split
        comm_info = {"layout": "2-way CFG split x %d-way frame sharding" % (world // 2) if cfg_split else "%d-way frame sharding" % world,
                     "fused_switches_per_forward": None if comm is None else getattr(comm, "fused_per_forward", None),
                     "impl": ("NVLink peer-memory exchange kernels (csrc/peer.cu), GroupNorm statistics fused into the frames->sites switch"
                              if isinstance(comm, _par.PeerFrameComm) else ("NCCL all_to_all_single + all_reduce" if comm is not None else "none (CFG split only)")),
                     "bytes_sent_per_forward_rank0": None if comm is None else int(getattr(comm, "bytes_per_forward", 0)),
                     "bytes_per_step": None if comm is None else int(getattr(comm, "bytes_per_forward", 0)) + int(dev["x_T"].numel() * 4),
                     "exposed_ms": None if comm is None else {"per_forward_rank0": getattr(comm, "exposed_ms", None), "eager_forward_ms": getattr(comm, "forward_ms", None),
                                                               "exchanges": getattr(comm, "n_exchanges", None),
                                                               "what": "device time of the in-stream exchange / statistics kernels of ONE eager forward on rank 0 "
                                                                       "(transfer + waiting for the slowest peer): not overlapped with compute"},
                     "cfg_exchange_bytes_per_step": int(dev["x_T"].numel() * 4) if cfg_split else 0}
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    if rank != 0:
        _finish(world, dist)
        return

    value = args.steps / float(t_dev)
    e2e_value = args.steps / float(t_e2e)
    line = {"metric": metric, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 (fp32 accumulate; fp32 norms/softmax/update)", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clk.summary(), "finite": finite,
            "step_tflops": {"achieved": 2 * UNET_FWD_TFLOP[args.workload] * value, "peak_sustained": peaks["tflops_sustained"],
                            "frac": 2 * UNET_FWD_TFLOP[args.workload] * value / peaks["tflops_sustained"],
                            "note": "reference-algorithm FLOPs (SURVEY.md 8d: %.2f TFLOP per U-Net forward) / measured step time" % UNET_FWD_TFLOP[args.workload]},
            "published_context": {"a100_readme_steps_per_s": A100_README_STEPS_PER_S[args.workload],
                                  "speedup_vs_a100_readme": value / A100_README_STEPS_PER_S[args.workload],
                                  "note": "README.md:117-122 (A100 40GB, whole-pipeline time / 50 steps); other hardware, so vs_baseline stays null"}}
    if world > 1:
        line["sharded_vs_single_max_err"] = shard_err
        line["comm"] = comm_info
    if world == 1:
        line.update(kernel_rooflines(wl, device, peaks))
        if not args.no_gpu_baseline:
            line["parity"], line["gpu_eager_baseline"] = gpu_parity_and_eager_baseline(wl, model, dev, sampler, run_step)
            line["vs_gpu_eager"] = {"value_ratio": value / line["gpu_eager_baseline"]["value"],
                                    "note": "this arm's device-resident steps/s / the eager-PyTorch reference algorithm on the same GPU"}
        if not args.no_vae:
            line["vae_decode"] = vae_decode_bench(wl, device)
        if not args.no_cpu_baseline:
            sd_cpu = {k: v.detach().float().cpu() for k, v in model.model.diffusion_model.state_dict().items()}
            del model, sampler
            torch.cuda.empty_cache()
            v, dt, cores, sample = cpu_frame_sample(wl, sd_cpu, 1, 1, args.workload)          # 2 samples: ~20-30 s of CPU work
            line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample, "estimated": True}
            line["cpu_baseline_config1"] = cpu_config1_measured(sd_cpu)
    print(json.dumps(line))
    _finish(world, dist)


def dump_outputs(out_dir, **arrays):
    """What a caller of the timed path received from its last step, one DIR/<name>.npy (float32) per array.  Weights, inputs and
    the per-step noise all come from fixed seeds, so two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.detach().float().cpu().numpy())


def _finish(world, dist):
    """End of a multi-rank run: every rank has its result; leave without tearing the process group down.  destroy_process_group() after
    NCCL collectives were captured into CUDA graphs hung at exit on the 4-GPU box (round 2, call C: the line was printed, the ranks never
    left), so the ranks meet at a barrier and exit hard."""
    sys.stdout.flush(); sys.stderr.flush()
    if world > 1:
        try:
            torch.cuda.synchronize()
            dist.barrier()
        except Exception:
            pass
        os._exit(0)


if __name__ == "__main__":
    main()
