"""Three-way (text + image) guidance as one batched U-Net forward on the GPU: the B=3 shared-prefix forward at full width against
three B=1 forwards, three sampler steps against the fp32 oracle, graph replay against eager, and (with >= 2 devices) a torchrun of
tools/multicond_check.py with the CFG split and with pure frame sharding, over the peer-memory kernels and over NCCL."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_ERR, MEAN_ERR = 0.02, 0.003


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _unet(over, seed):
    from oracle import synth
    from viewcrafter_b200.configs import UNET_PARAMS
    from viewcrafter_b200.unet import UNetModel
    m = UNetModel(**dict(UNET_PARAMS, **over))
    m.load_state_dict(synth.synth_state_dict(synth.module_shapes(m), seed), strict=True)
    return m.cuda().eval()


def test_three_branch_shared_prefix_full_width_vs_single_forwards():
    """model_channels=320 (the shipped widths): B=3 with the prefix computed once vs the three B=1 forwards of the same branches.
    Within fp16 rounding, not bit-exact: a B=3 GEMM / GroupNorm launches other tile and split counts than B=1 ones (and GroupNorm
    sums with shared-memory float atomics), so the fp32 accumulations round to fp16 differently.  Measured on a B200: max 0.0044,
    mean 0.00084 -- the plain B=3 forward without the hint differs from the B=1 forwards by the same amount (max 0.0047)."""
    _need_gpu()
    from viewcrafter_b200.unet import SHARED_PREFIX_ANY_LAYOUT
    m = _unet({}, 12)
    g = torch.Generator().manual_seed(13)
    x1 = torch.randn(1, 8, 3, 8, 16, generator=g).cuda()
    t1, fs1 = torch.tensor([499]).cuda(), torch.tensor([10]).cuda()
    ctxs = [torch.randn(1, 333, 1024, generator=g).cuda() for _ in range(3)]
    singles = torch.cat([m(x1, t1, context=c, fs=fs1) for c in ctxs], 0)
    X, Tt, F, C = x1.repeat(3, 1, 1, 1, 1), t1.repeat(3), fs1.repeat(3), torch.cat(ctxs, 0)
    plain = m(X, Tt, context=C, fs=F)
    for hint in (True, SHARED_PREFIX_ANY_LAYOUT):
        y = m(X, Tt, context=C, fs=F, cfg_shared_prefix=hint)
        err, err_plain = (y - singles).abs(), (plain - singles).abs()
        print(f"B=3 shared prefix ({hint!r}) vs 3 x B=1: bit-exact {torch.equal(y, singles)}, max {float(err.max()):.4g} mean {float(err.mean()):.4g}; "
              f"plain B=3 vs 3 x B=1: max {float(err_plain.max()):.4g}")
        assert float(err.max()) <= MAX_ERR and float(err.mean()) <= MEAN_ERR
    assert float((singles[0] - singles[2]).abs().mean()) > 10 * MEAN_ERR


@pytest.mark.parametrize("batch_cfg", [False, True])
def test_multicond_sample_three_steps_vs_oracle(batch_cfg):
    """ddim_multiplecond.DDIMSampler.sample (S=3, eta=1, CFG 7.5, cfg_img 2.5, rescale 0.7) with identical x_T and per-step noise on
    both sides; batch_cfg=True runs each step as ONE B=3 forward with the shared prefix."""
    _need_gpu()
    from oracle import lvdm_oracle as O
    from oracle import synth
    from viewcrafter_b200.configs import UNET_PARAMS
    from viewcrafter_b200.ddim_multiplecond import DDIMSampler
    from viewcrafter_b200.diffusion import LatentDiffusion
    model = LatentDiffusion(dict(UNET_PARAMS, model_channels=64), None, base_scale=0.7)
    unet = model.model.diffusion_model
    sd = synth.synth_state_dict(synth.module_shapes(unet), seed=41)
    unet.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    g = torch.Generator().manual_seed(42)
    T, H, W, S = 5, 8, 8, 3
    shape = (1, 4, T, H, W)
    x_T, cc = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
    ctx_c, ctx_u, ctx_i = (torch.randn(1, 333, 1024, generator=g) for _ in range(3))
    fs = torch.tensor([10])
    ccg = cc.cuda()
    c, uc, uc_img = ({"c_crossattn": [k.cuda()], "c_concat": [ccg]} for k in (ctx_c, ctx_u, ctx_i))
    batches = []
    real_forward = unet.forward
    unet.forward = lambda xx, *a, **k: (batches.append(xx.shape[0]), real_forward(xx, *a, **k))[1]
    sampler = DDIMSampler(model, batch_cfg=batch_cfg)
    torch.manual_seed(43)
    out, inter = sampler.sample(S=S, batch_size=1, shape=shape[1:], conditioning=c, eta=1.0, verbose=False, x_T=x_T.cuda(),
                                unconditional_guidance_scale=7.5, unconditional_conditioning=uc, fs=fs.cuda(), cfg_img=2.5,
                                unconditional_conditioning_img_nonetext=uc_img, timestep_spacing="uniform_trailing", guidance_rescale=0.7)
    torch.manual_seed(43)
    noises = [torch.randn(shape, device="cuda").cpu() for _ in range(S)]
    sched = O.model_schedule(base_scale=0.7)

    def model_fn(x, t, cond):
        with torch.no_grad():
            return O.unet_forward(sd, torch.cat([x, cc], 1), t, cond, fs)

    ref, ref_inter = O.ddim_sample(model_fn, sched, shape, S, ctx_c, ctx_u, x_T, noises, fixed_prev_scale=False, uncond_img=ctx_i, cfg_img=2.5)
    err = (out.cpu() - ref).abs()
    print(f"three-way ddim S=3 batch_cfg={batch_cfg}: max err {float(err.max()):.4g} mean {float(err.mean()):.4g} ref std {float(ref.std()):.3g}")
    assert batches == ([3] * S if batch_cfg else [1] * (3 * S))
    assert len(inter["x_inter"]) == len(ref_inter["x_inter"])
    assert float(err.max()) <= 0.15 and float(err.mean()) <= 0.02      # CFG 7.5 amplifies the fp16 U-Net error ~16x (two-way test)


def test_three_branch_graph_replay_equals_eager():
    """enable_cuda_graph() with the B=3 shared-prefix batch: call 1 eager, call 2 capture, calls 3+ replay -- bit-identical to eager
    forwards of the same inputs; the B=3 prefix graph is keyed apart from a B=3 forward without the hint."""
    _need_gpu()
    from viewcrafter_b200.unet import SHARED_PREFIX_ANY_LAYOUT
    m = _unet(dict(model_channels=64), 31)
    g = torch.Generator().manual_seed(32)
    ctx = torch.randn(3, 333, 1024, generator=g).cuda()
    fs = torch.tensor([10, 10, 10]).cuda()
    xs = [torch.randn(1, 8, 5, 8, 16, generator=g).cuda().repeat(3, 1, 1, 1, 1) for _ in range(4)]
    ts = [torch.tensor([t] * 3).cuda() for t in (999, 979, 499, 19)]
    eager = [m(x, t, context=ctx, fs=fs, cfg_shared_prefix=SHARED_PREFIX_ANY_LAYOUT) for x, t in zip(xs, ts)]
    m.enable_cuda_graph()
    for i, (x, t) in enumerate(zip(xs, ts)):
        y = m(x, t, context=ctx, fs=fs, cfg_shared_prefix=SHARED_PREFIX_ANY_LAYOUT)
        assert torch.equal(y, eager[i]), (i, float((y - eager[i]).abs().max()))
    plain = [m(xs[0], ts[0], context=ctx, fs=fs) for _ in range(3)]
    keys = [k for k, e in m._graphs.items() if e["graph"] is not None]
    assert len(keys) == 2 and len({k[5] for k in keys}) == 2                # the flag value is part of the graph key
    m.enable_cuda_graph(False)
    ref_plain = m(xs[0], ts[0], context=ctx, fs=fs)
    assert all(torch.equal(p, ref_plain) for p in plain)


@pytest.mark.parametrize("cfg_split", [True, False])
@pytest.mark.parametrize("peer", ["1", "0"])
def test_three_way_step_on_two_gpus(cfg_split, peer):
    """tools/multicond_check.py on 2 ranks: CFG split (B=2 + B=1) or pure frame sharding (B=3 per rank); peer-memory kernels or NCCL."""
    world = 2
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} CUDA devices")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(ROOT, "tools", "multicond_check.py")] + ([] if cfg_split else ["--no-cfg-split"])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=800, env=dict(os.environ, VC_PEER_COMM=peer))
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and "MULTICOND_CHECK_OK" in r.stdout
