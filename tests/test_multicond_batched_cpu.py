"""Three-way (text + image) guidance as one batched U-Net forward, on the CPU op double (tests/fake_ops.py):
  * the B=3 shared-prefix forward against three independent B=1 forwards;
  * the three-way sampler with batch_cfg=True (one U-Net call per step, the stacked conditioning built once) against the
    reference golden ddim_multicond_small.npz;
  * gloo runs of a three-way DDIM step under parallel.shard_model (CFG split x frame sharding, pure frame sharding at B=3 per rank)
    against the single-process step;
  * the peer-memory pieces that index samples at B=3 / 4: the fused epilogue scatter routing and the statistics slot layout."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import synth
from tests import fake_ops
from tests import test_peer_scatter_model_cpu as scatter_model
from viewcrafter_b200.configs import UNET_PARAMS
from viewcrafter_b200.parallel import frame_ranges


@pytest.fixture
def cpu_ops(monkeypatch):
    fake_ops.install(monkeypatch)
    return fake_ops


@pytest.mark.parametrize("hint", [True, "any_layout"])
def test_three_branch_shared_prefix_equals_three_single_forwards(cpu_ops, hint):
    """SURVEY.md App. C.2 for three branches: the context-free prefix runs once at B=1 and is replicated to B=3 before the first
    cross-attention; every branch equals its own B=1 forward.  Not bit-equal on this double: its CPU GEMMs / convolutions round
    differently at B=3 and B=1 (a plain B=3 forward without the hint differs from the B=1 forwards by the same ~5e-3), so the
    tolerance is that of test_shared_cfg_prefix_and_kv_cache."""
    from viewcrafter_b200.unet import SHARED_PREFIX_ANY_LAYOUT, UNetModel
    assert SHARED_PREFIX_ANY_LAYOUT == "any_layout"
    m = UNetModel(**dict(UNET_PARAMS, model_channels=64)).eval()
    m.load_state_dict(synth.synth_state_dict(synth.module_shapes(m), seed=61), strict=True)
    g = torch.Generator().manual_seed(62)
    x1 = torch.randn(1, 8, 3, 8, 8, generator=g)
    t1, fs1 = torch.tensor([499]), torch.tensor([10])
    ctxs = [torch.randn(1, 333, 1024, generator=g) for _ in range(3)]
    singles = [m(x1, t1, context=c, fs=fs1) for c in ctxs]
    calls = []
    real_spatial = UNetModel._spatial_tf

    def spy(P, h, ctx, B, T, H, W, expand=False, out_plan=None):
        calls.append((h.shape[0], B, expand))
        return real_spatial(P, h, ctx, B, T, H, W, expand=expand, out_plan=out_plan)

    UNetModel._spatial_tf = staticmethod(spy)
    try:
        y = m(x1.repeat(3, 1, 1, 1, 1), t1.repeat(3), context=torch.cat(ctxs, 0), fs=fs1.repeat(3), cfg_shared_prefix=hint)
    finally:
        UNetModel._spatial_tf = staticmethod(real_spatial)
    assert calls[0] == (3 * 8 * 8, 3, True)                 # the first SpatialTransformer gets ONE batch element and expands it
    assert all(not e for _, _, e in calls[1:])
    for b in range(3):
        d = (y[b:b + 1] - singles[b]).abs()
        assert float(d.max()) < 0.02 and float(d.mean()) < 3e-3, (b, float(d.max()), float(d.mean()))
        assert float((singles[b] - singles[(b + 1) % 3]).abs().mean()) > 5 * float(d.mean())      # the branches do differ


def _toy_model(golden, calls, contexts):
    """The reference golden's toy denoiser, batched: one row per stacked branch (c['k'] / c['b'] are lists like c_crossattn)."""
    from viewcrafter_b200.diffusion import LatentDiffusion
    model = LatentDiffusion(dict(UNET_PARAMS, model_channels=64), None, base_scale=0.3).eval()

    def toy(x, t, c, **kw):
        calls.append((x.shape[0], kw.get("cfg_shared_prefix")))
        contexts.append(c["b"][0])
        k = c["k"][0].reshape(-1, 1, 1, 1, 1)
        return torch.tanh(0.7 * x * k + 0.05 * torch.sin(t.float())[:, None, None, None, None]) + 0.1 * c["b"][0]

    model.apply_model = toy
    return model


@pytest.mark.parametrize("tag,S,cfg_img", [("S5", 5, 2.5), ("S8", 8, None)])
def test_batched_multicond_sampler_matches_reference_golden(cpu_ops, golden_dir, tag, S, cfg_img):
    """batch_cfg=True: ONE apply_model call per step at B=3 (cond, uncond, image-only), the stacked conditioning is the same
    tensor every step, the prefix hint is sent when the branches share c_concat, and the samples are the reference sampler's."""
    from viewcrafter_b200.ddim_multiplecond import DDIMSampler
    from viewcrafter_b200.unet import SHARED_PREFIX_ANY_LAYOUT
    import viewcrafter_b200.ddim_multiplecond as mod
    g = np.load(os.path.join(golden_dir, "ddim_multicond_small.npz"))
    calls, contexts = [], []
    model = _toy_model(g, calls, contexts)
    noises = iter(torch.from_numpy(g[f"{tag}_noises"]))
    cc = torch.zeros(1, 4, 3, 4, 6)
    cond = {"k": [torch.tensor([1.3])], "b": [torch.from_numpy(g[f"{tag}_cond_b"])], "c_concat": [cc]}
    unc = {"k": [torch.tensor([0.4])], "b": [torch.from_numpy(g[f"{tag}_uncond_b"])], "c_concat": [cc]}
    unc_img = {"k": [torch.tensor([0.9])], "b": [torch.from_numpy(g[f"{tag}_uncond_img_b"])], "c_concat": [cc]}
    real_randn = torch.randn
    try:
        mod.torch.randn = lambda shape, device=None: next(noises)
        smp = DDIMSampler(model, batch_cfg=True)
        out, inter = smp.sample(S=S, batch_size=1, shape=(4, 3, 4, 6), conditioning=cond, eta=1.0, verbose=False,
                                x_T=torch.from_numpy(g[f"{tag}_x_T"]), unconditional_guidance_scale=7.5,
                                unconditional_conditioning=unc, timestep_spacing="uniform_trailing", guidance_rescale=0.7,
                                cfg_img=cfg_img, unconditional_conditioning_img_nonetext=unc_img)
    finally:
        mod.torch.randn = real_randn
    assert calls == [(3, SHARED_PREFIX_ANY_LAYOUT)] * S
    assert all(c is contexts[0] for c in contexts)                    # one canonical stacked context per clip
    np.testing.assert_allclose(out.numpy(), g[f"{tag}_samples"], rtol=0, atol=5e-5)
    np.testing.assert_allclose(inter["pred_x0"][-1].numpy(), g[f"{tag}_pred_x0_last"], rtol=0, atol=5e-5)


def test_batched_multicond_keeps_separate_calls_when_not_stackable(cpu_ops, golden_dir):
    """Conditioning dicts with different keys cannot be stacked: the reference's three calls remain."""
    from viewcrafter_b200.ddim_multiplecond import DDIMSampler
    g = np.load(os.path.join(golden_dir, "ddim_multicond_small.npz"))
    calls, contexts = [], []
    model = _toy_model(g, calls, contexts)
    b = torch.from_numpy(g["S5_cond_b"])
    cond = {"k": [torch.tensor([1.3])], "b": [b]}
    unc = {"k": [torch.tensor([0.4])], "b": [b], "extra": [b]}
    smp = DDIMSampler(model, batch_cfg=True)
    smp.sample(S=2, batch_size=1, shape=(4, 3, 4, 6), conditioning=cond, eta=1.0, verbose=False, unconditional_guidance_scale=7.5,
               unconditional_conditioning=unc, timestep_spacing="uniform_trailing", unconditional_conditioning_img_nonetext=cond)
    assert [n for n, _ in calls] == [1] * 6


# ------------------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, cfg_split, H, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    import _pytest.monkeypatch as mpatch
    from viewcrafter_b200 import parallel
    from viewcrafter_b200.ddim_multiplecond import DDIMSampler
    from viewcrafter_b200.diffusion import LatentDiffusion
    mpx = mpatch.MonkeyPatch()
    fake_ops.install(mpx)
    model = LatentDiffusion(dict(UNET_PARAMS, model_channels=64), None, base_scale=0.3).eval()
    unet = model.model.diffusion_model
    unet.load_state_dict(synth.synth_state_dict(synth.module_shapes(unet), 7), strict=True)
    g = torch.Generator().manual_seed(8)
    shape = (1, 4, 4, H, 16)
    x, cc = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
    c = {"c_crossattn": [torch.randn(1, 333, 1024, generator=g)], "c_concat": [cc]}
    uc = {"c_crossattn": [torch.randn(1, 333, 1024, generator=g)], "c_concat": [cc]}
    uc_img = {"c_crossattn": [torch.randn(1, 333, 1024, generator=g)], "c_concat": [cc]}
    ts = torch.full((1,), 599, dtype=torch.long)
    batches = []
    real_forward = unet.forward
    unet.forward = lambda xx, *a, **k: (batches.append(xx.shape[0]), real_forward(xx, *a, **k))[1]

    def step():
        smp = DDIMSampler(model, batch_cfg=True)
        smp.make_schedule(5, "uniform_trailing", 1.0, verbose=False)
        torch.manual_seed(9)
        return smp.p_sample_ddim(x, c, ts, index=2, unconditional_guidance_scale=7.5, unconditional_conditioning=uc, cfg_img=5.0,
                                 unconditional_conditioning_img_nonetext=uc_img, fs=torch.tensor([10]), guidance_rescale=0.7)[0]

    ref = step()
    assert batches == [3]
    batches.clear()
    parallel.shard_model(model, dist, rank, world, cfg_split=cfg_split)
    out = step()
    cfg = getattr(model, "_cfg", None)
    q.put((rank, float((out - ref).abs().max()), list(batches), None if cfg is None else cfg.branch))
    dist.barrier()
    dist.destroy_process_group()
    mpx.undo()


def _spawn(world, cfg_split, H):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cfg_split, H, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=900)
        assert p.exitcode == 0, f"rank exited with {p.exitcode}"
    return sorted(q.get(timeout=10) for _ in range(world))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_three_way_step_cfg_split_matches_single_process(world):
    """world 2 = CFG split 1+1 (rank 0: cond + image-only at B=2 with the shared prefix, rank 1: uncond); world 4 / 8 = the same
    split x 2- / 4-way frame sharding (the branch-0 prefix runs frame-sharded at B=1)."""
    res = _spawn(world, True, 16)
    for rank, d, batches, branch in res:
        assert branch == (0 if rank < world // 2 else 1)
        assert batches == ([2] if branch == 0 else [1]), (rank, batches)
        # the reference step runs one B=3 forward, the split a B=2 and a B=1 one (the double rounds differently per batch size, see
        # above), and frame sharding regroups the 5-D GroupNorm sums: fp16 noise amplified by CFG, as in test_parallel_cpu.py
        assert d < 0.15, (rank, d)


@pytest.mark.parametrize("world,H", [(2, 16), (3, 24)])
def test_three_way_step_frame_sharded_b3_matches_single_process(world, H):
    """cfg_split=False: every rank runs the B=3 forward with the shared prefix on its frames (H*W divisible by the world size at
    every level: 24 x 16 for three ranks)."""
    res = _spawn(world, False, H)
    for rank, d, batches, branch in res:
        assert branch is None and batches == [3], (rank, batches)
        assert d < 0.15, (rank, d)


# ------------------------------------------------------------------------------------------------------------------------------
def _plan_accepts(P, T, B, HW):
    """PeerFrameComm.scatter_plan's rank / frame alignment rule (the shape part of it)."""
    return all(f1 > f0 and (B == 1 or ((f1 - f0) * HW) % 128 == 0) for f0, f1 in frame_ranges(T, P))


@pytest.mark.parametrize("P,T,B,H,W,geom", [
    (2, 25, 3, 36, 64, "conv"), (2, 5, 3, 16, 16, "conv"), (4, 8, 3, 16, 32, "conv"), (2, 5, 3, 16, 16, "linear"),
    (4, 7, 3, 16, 32, "linear"), (2, 25, 3, 36, 64, "linear"), (2, 5, 4, 16, 16, "conv"), (2, 5, 4, 16, 16, "linear"),
])
def test_frames_to_sites_routing_three_samples(P, T, B, H, W, geom):
    """The epilogue scatter of the B=3 three-way forward (and B=4, the new Bmax) on the shapes scatter_plan accepts."""
    assert _plan_accepts(P, T, B, H * W)
    scatter_model.test_frames_to_sites_routing_equals_the_layout_permutation(P, T, B, H, W, geom)


@pytest.mark.parametrize("P,T,B,HW,geom", [
    (2, 25, 3, 2304, "tconv"), (2, 5, 3, 256, "tconv"), (2, 5, 3, 256, "linear"), (4, 7, 3, 512, "linear"), (4, 8, 3, 512, "tconv"),
    (2, 25, 3, 2304, "linear"), (2, 5, 4, 256, "tconv"),
])
def test_sites_to_frames_routing_three_samples(P, T, B, HW, geom):
    assert _plan_accepts(P, T, B, HW)
    scatter_model.test_sites_to_frames_routing_equals_the_layout_permutation(P, T, B, HW, geom)


def test_plan_rule_rejects_unaligned_sample_boundaries():
    """At B > 1 a 128-row m-tile must not span two samples of one rank: 13 frames x 18 x 32 pixels is not a multiple of 128."""
    assert not _plan_accepts(2, 25, 3, 18 * 32)
    assert _plan_accepts(2, 25, 1, 18 * 32)


# ------------------------------------------------------------------------------------------------------------------------------
def _peer_finish_publish(world, Bmax, B, threads, strided=True):
    """csrc/peer.cu peer_finish, publish step: which (writer rank, slot) pairs every rank's slot array receives.  Returns
    {reader rank: list of slot indices written into its array}; `strided` False models the former one-thread-per-value code."""
    parity = 1
    written = {q: [] for q in range(world)}
    for me in range(world):
        for tid in range(threads):
            idx = range(tid, B * 64, threads) if strided else ([tid] if tid < B * 64 else [])
            for i in idx:
                b, t = i >> 6, i & 63
                slot = ((parity * Bmax + b) * world + me) * 64 + t
                for q in range(world):
                    written[q].append(slot)
    return written


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("B", [3, 4])
def test_peer_finish_publishes_every_sample_group_once(world, B):
    """With the 128-thread all-reduce block (and the 256..512-thread exchange blocks) every (sample, group, sum|sumsq) value of every
    rank lands exactly once in every rank's slots, inside the [2][Bmax][world][64] array, and the gather of the first B*world*64
    values of the parity half is complete."""
    Bmax = 4
    for threads in (128, 256, 480, 512):
        written = _peer_finish_publish(world, Bmax, B, threads)
        for q in range(world):
            slots = sorted(written[q])
            assert len(slots) == len(set(slots)) == B * world * 64
            assert max(slots) < 2 * Bmax * world * 64
            base = 1 * Bmax * world * 64
            assert slots == list(range(base, base + B * world * 64))         # exactly what cur_stats gathers
    # the former indexing (tid < B*64 publishes one value) misses samples 2.. with a 128-thread block
    assert len(_peer_finish_publish(world, Bmax, B, 128, strided=False)[0]) == 2 * world * 64
