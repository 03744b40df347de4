"""torchrun target: one three-way-guidance DDIM step (text + image CFG, ddim_multiplecond.DDIMSampler with batch_cfg=True) under
parallel.shard_model vs the single-GPU step (rank 0 prints, MULTICOND_CHECK_OK on success).

  default        CFG split (even world): branch-0 ranks run (cond, image-only) as one B=2 forward with the shared prefix, branch-1 ranks
                 uncond at B=1, CfgComm.exchange3 hands every rank all three predictions
  --no-cfg-split pure frame sharding: every rank runs the B=3 forward with the shared prefix on its frames

VC_PEER_COMM=1 (default) also checks the NVLink peer-memory exchange at B=3 and B=4 samples per rank (layout switch, GroupNorm
statistics published by peer_finish for every sample) against the NCCL implementation over all ranks; VC_PEER_COMM=0 runs NCCL only.
The step is repeated with the U-Net replayed as a captured CUDA graph."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

ap = argparse.ArgumentParser()
ap.add_argument("--no-cfg-split", action="store_true")
args = ap.parse_args()
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from oracle import synth
from viewcrafter_b200 import parallel
from viewcrafter_b200.configs import UNET_PARAMS
from viewcrafter_b200.ddim_multiplecond import DDIMSampler
from viewcrafter_b200.diffusion import LatentDiffusion

peer = os.environ.get("VC_PEER_COMM", "1") != "0"
ok = True
T = 5

# ---- peer-memory exchange at B=3 / 4 samples per rank vs the NCCL collectives ----
if peer:
    pc = parallel.PeerFrameComm(dist, rank, world, None, torch.device("cuda", local))
    rc = parallel.FrameComm(dist, rank, world, None)
    f0, f1 = pc.bind(T)
    rc.bind(T)
    for Bq, HWq, Cq in ((3, 256, 64), (3, 64, 320), (4, 16, 1280), (3, 1024, 640)):
        gq = torch.Generator().manual_seed(200 + rank)
        hq = (torch.randn(Bq * (f1 - f0) * HWq, Cq, generator=gq) * 1.5 + 0.3).half().cuda()
        # give every sample its own mean / scale, so that a sample whose statistics were not published shows up
        hq = (hq.view(Bq, -1, Cq) * torch.tensor([1.0, 2.0, 0.5, 3.0][:Bq], device="cuda").view(Bq, 1, 1).half()
              + torch.tensor([0.0, 1.0, -2.0, 0.5][:Bq], device="cuda").view(Bq, 1, 1).half()).reshape(-1, Cq).contiguous()
        a = pc.to_sites(hq, Bq, HWq)
        b = rc.to_sites(hq, Bq, HWq)
        same = torch.equal(a, b)
        gam, bet = torch.rand(Cq, device="cuda") + 0.5, torch.randn(Cq, device="cuda") * 0.1
        n1 = pc.groupnorm5d(a, Bq, gam, bet, 1e-5, True, T * HWq, True)             # statistics that rode on the exchange
        n2 = rc.groupnorm5d(b, Bq, gam, bet, 1e-5, True, T * HWq, True)
        n3 = pc.groupnorm5d(b.clone(), Bq, gam, bet, 1e-5, True, T * HWq, False)    # vc_peer_groupnorm_stats
        e12, e13 = float((n1.float() - n2.float()).abs().max()), float((n3.float() - n2.float()).abs().max())
        back = pc.to_frames(a.clone(), Bq, HWq)
        rt = torch.equal(back, hq)
        torch.cuda.synchronize()
        good = same and rt and e12 < 4e-3 and e13 < 4e-3
        ok = ok and good
        print(f"[rank {rank}] peer exchange B={Bq} HW={HWq} C={Cq}: to_sites==nccl {same}, round trip {rt}, "
              f"GN(fused stats) err {e12:.2e}, GN(peer stats) err {e13:.2e}", flush=True)
    dist.barrier()
    pc.close()

# ---- the three-way step ----
with torch.device("cuda"):
    model = LatentDiffusion(dict(UNET_PARAMS, model_channels=64), None, base_scale=0.3).eval()
unet = model.model.diffusion_model
unet.load_state_dict(synth.synth_state_dict(synth.module_shapes(unet), 7), strict=True)
unet._packed = None
g = torch.Generator().manual_seed(8)
shape = (1, 4, T, 16, 16)
xs, cc = torch.randn(shape, generator=g).cuda(), torch.randn(shape, generator=g).cuda()
ctx = lambda: {"c_crossattn": [torch.randn(1, 333, 1024, generator=g).cuda()], "c_concat": [cc]}
c, uc, uc_img = ctx(), ctx(), ctx()
ts = torch.full((1,), 599, dtype=torch.long, device="cuda")
smp = DDIMSampler(model, batch_cfg=True)
smp.make_schedule(5, "uniform_trailing", 1.0, verbose=False)


def step():
    torch.manual_seed(9)
    return smp.p_sample_ddim(xs, c, ts, index=2, unconditional_guidance_scale=7.5, unconditional_conditioning=uc, cfg_img=7.5,
                             unconditional_conditioning_img_nonetext=uc_img, fs=torch.tensor([10], device="cuda"), guidance_rescale=0.7)[0]


ref = step()
comm = parallel.shard_model(model, dist, rank, world, cfg_split=not args.no_cfg_split)
split = getattr(model, "_cfg", None) is not None
outs = [step() for _ in range(2)]
unet.enable_cuda_graph()
graphed = [step() for _ in range(3)]                  # eager, capture, replay
unet.enable_cuda_graph(False)
torch.cuda.synchronize()
d = torch.tensor([float((o - ref).abs().max()) for o in outs] + [float((o - outs[0]).abs().max()) for o in graphed], device="cuda")
dist.all_reduce(d, op=dist.ReduceOp.MAX)
d_single, d_graph = float(d[:2].max()), float(d[2:].max())
# the single-GPU step runs one B=3 forward, the split a B=2 and a B=1 one (other tile / split counts, other fp16 roundings), GroupNorm's
# shared-memory float atomics sum in a run-dependent order and frame sharding regroups the 5-D GroupNorm sums; the guidance
# (1 + 7.5 + 7.5) amplifies all of it (the sharded tolerance of tools/parallel_check.py)
tol = 0.15
ok = ok and d_single < tol and d_graph < tol
flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
ok = bool(flag.item() > 0)
if rank == 0:
    layout = f"CFG split 2 x {world // 2} frames" if split else f"{world}-way frames, B=3 per rank"
    print(f"world {world} ({layout}, {type(comm).__name__ if comm else 'no frame comm'}): three-way step |sharded - single| {d_single:.4g}, "
          f"graph replay vs eager {d_graph:.4g}, switches fused into GEMM epilogues {getattr(comm, 'fused_switches', 0)}")
    if ok:
        print("MULTICOND_CHECK_OK")
# leave like bench.py does: destroy_process_group() after NCCL collectives were captured into CUDA graphs (VC_PEER_COMM=0) can hang
sys.stdout.flush(); sys.stderr.flush()
torch.cuda.synchronize()
dist.barrier()
os._exit(0 if ok else 1)
