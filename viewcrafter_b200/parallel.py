"""Frame-sharded multi-GPU execution of the U-Net forward (one process per GPU, torch.distributed / NCCL over NVLink).

SURVEY.md 8(e): every spatial op (2-D convs, per-frame GroupNorm, SpatialTransformer incl. attention, Down/Upsample)
is independent per frame, so rank r owns a contiguous range of the T frames.  The ops that couple frames --
TemporalTransformer (17 per forward) and TemporalConvBlock (22 per forward), including their 5-D GroupNorm statistics
-- run in the transposed "site" layout: every rank holds ALL T frames of H*W/P pixels (H*W is divisible by 8 at every
level), which is perfectly balanced.  The two layouts are exchanged with ONE uneven all-to-all each way
(NCCL all_to_all_single over NVSwitch; volume per rank = activation_bytes * (P-1)/P^2) and the 5-D GroupNorm adds a
[B,32,2] all-reduce.  The reference has no multi-GPU path for this (SURVEY.md 2a); this is new functionality.
"""
from __future__ import annotations

import os
from typing import List

import torch


def frame_ranges(T: int, world: int) -> List[tuple]:
    """Contiguous, as-even-as-possible split of T frames: 25 over 8 -> 4,3,3,3,3,3,3,3."""
    base, extra = divmod(T, world)
    out, f = [], 0
    for r in range(world):
        n = base + (1 if r < extra else 0)
        out.append((f, f + n))
        f += n
    return out


class FrameComm:
    def __init__(self, dist, rank: int, world: int, group=None):
        self.dist, self.rank, self.world, self.group = dist, rank, world, group
        self.T = None
        self.ranges = None
        self.bytes_moved = 0            # all-to-all payload sent by this rank (for the bench report)
        self._prof = None               # list of (start, end) CUDA events around every exchange when profiling (bench.py: exposed comm time)

    def __bool__(self):
        return self.world > 1

    def bind(self, T: int):
        self.T = T
        self.ranges = frame_ranges(T, self.world)
        return self.ranges[self.rank]

    # -- exposed-communication profile: the exchanges run in-stream, so their device time (incl. waiting for the peers) is exposed --
    def profile(self, on: bool):
        self._prof = [] if on else None

    def profile_ms(self) -> float:
        torch.cuda.synchronize()
        return float(sum(a.elapsed_time(b) for a, b in (self._prof or [])))

    def _mark(self):
        if self._prof is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _done(self, e0):
        if e0 is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            self._prof.append((e0, e1))

    # -- layout transposes -----------------------------------------------------------------------
    def to_sites(self, h: torch.Tensor, B: int, HW: int) -> torch.Tensor:
        e0 = self._mark()
        out = self._to_sites(h, B, HW)
        self._done(e0)
        return out

    def to_frames(self, t: torch.Tensor, B: int, HW: int) -> torch.Tensor:
        e0 = self._mark()
        out = self._to_frames(t, B, HW)
        self._done(e0)
        return out

    def _to_sites(self, h: torch.Tensor, B: int, HW: int) -> torch.Tensor:
        """[(b, t_local, hw), C] -> [(b, t_all, hw_local), C]."""
        P, C = self.world, h.shape[1]
        assert HW % P == 0, f"H*W={HW} must be divisible by the world size {P}"
        HWl = HW // P
        Tl = self.ranges[self.rank][1] - self.ranges[self.rank][0]
        send = h.view(B, Tl, P, HWl, C).permute(2, 0, 1, 3, 4).contiguous().view(P * B * Tl * HWl, C)
        out_rows = [B * (f1 - f0) * HWl for f0, f1 in self.ranges]
        recv = torch.empty((sum(out_rows), C), device=h.device, dtype=h.dtype)
        self.dist.all_to_all_single(recv, send, output_split_sizes=out_rows, input_split_sizes=[B * Tl * HWl] * P, group=self.group)
        self.bytes_moved += send.numel() * send.element_size() * (P - 1) // P
        if B == 1:
            return recv                                                   # chunks arrive in frame order already
        parts = [c.view(B, -1, HWl, C) for c in torch.split(recv, out_rows, 0)]
        return torch.cat(parts, dim=1).reshape(B * self.T * HWl, C)

    def _to_frames(self, t: torch.Tensor, B: int, HW: int) -> torch.Tensor:
        """[(b, t_all, hw_local), C] -> [(b, t_local, hw), C]."""
        P, C = self.world, t.shape[1]
        HWl = HW // P
        Tl = self.ranges[self.rank][1] - self.ranges[self.rank][0]
        in_rows = [B * (f1 - f0) * HWl for f0, f1 in self.ranges]
        if B == 1:
            send = t
        else:
            t4 = t.view(B, self.T, HWl, C)
            send = torch.cat([t4[:, f0:f1].reshape(-1, C) for f0, f1 in self.ranges], 0)
        recv = torch.empty((P * B * Tl * HWl, C), device=t.device, dtype=t.dtype)
        self.dist.all_to_all_single(recv, send.contiguous(), output_split_sizes=[B * Tl * HWl] * P, input_split_sizes=in_rows, group=self.group)
        self.bytes_moved += (send.numel() - in_rows[self.rank] * C) * send.element_size()
        return recv.view(P, B, Tl, HWl, C).permute(1, 2, 0, 3, 4).contiguous().view(B * Tl * HW, C)

    def all_reduce(self, t: torch.Tensor):
        self.dist.all_reduce(t, group=self.group)

    def scatter_plan(self, to_sites: bool, B: int, HW: int, Cc: int):
        """No fused switch with NCCL collectives (see PeerFrameComm.scatter_plan): the caller switches separately."""
        return None

    def groupnorm5d(self, x, B, gamma, beta, eps, silu, stat_rows, fresh: bool):
        """GroupNorm(32) of a site-layout tensor whose statistics span the ranks of the group.  `fresh`: x is the tensor the
        last to_sites() returned (the peer-memory path already holds its statistics)."""
        from . import ops
        st = ops.groupnorm_stats(x, B)
        e0 = self._mark()
        self.all_reduce(st)
        self._done(e0)
        return ops.groupnorm_apply(x, B, st, stat_rows, gamma, beta, eps, silu)

    def gather_frames(self, y_local: torch.Tensor, T: int) -> torch.Tensor:
        """[B,C,T_local,H,W] per rank -> the full [B,C,T,H,W] on every rank (3.7 MB at the headline size)."""
        B, C, _, H, W = y_local.shape
        tmax = max(f1 - f0 for f0, f1 in self.ranges)
        mine = y_local.new_zeros((B, C, tmax, H, W))
        mine[:, :, :y_local.shape[2]] = y_local
        parts = y_local.new_empty((self.world, B, C, tmax, H, W))
        self.dist.all_gather_into_tensor(parts.view(-1), mine.view(-1), group=self.group)       # uneven frame counts: padded to the largest shard
        return torch.cat([parts[r, :, :, :f1 - f0] for r, (f0, f1) in enumerate(self.ranges)], dim=2)


class PeerFrameComm(FrameComm):
    """FrameComm whose layout switches and GroupNorm statistics run as this library's own kernels over NVLink peer memory
    (csrc/peer.cu) instead of NCCL collectives: every rank maps the receive buffers, flag words and statistics slots of the
    other ranks of its group (CUDA IPC: cudaMalloc'd buffers, handles exchanged once over the process group, opened with the
    importing rank's compute device current) and
      * to_sites / to_frames are ONE kernel each (rows stored straight into the owning rank's buffer; no pack / unpack copy),
      * the statistics of the 5-D GroupNorm that follows every to_sites ride along with it (no statistics pass, no all-reduce),
      * the GroupNorms in the middle of a temporal block exchange 2 x 32 floats per sample through the same flag protocol.
    Up to `bmax` (<= 4) batch samples per rank: the three branches of three-way guidance run as one B=3 forward.
    The receive buffers are reused by every switch (one per direction): tensors returned by to_sites()/to_frames() are views
    of them and are only valid until the next switch in the same direction -- UNetModel clones the ones it keeps as skips."""

    def __init__(self, dist, rank: int, world: int, group, device, bmax: int = 4):
        super().__init__(dist, rank, world, group)
        from . import _lib
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.bmax = bmax
        self._bufs = {}            # name -> (own tensor, [device pointer of rank q's buffer as mapped here], capacity in elements)
        self._own_ptrs, self._peer_ptrs = [], []
        with torch.cuda.device(self.device):
            self.seq = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.done = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.cur_stats = torch.zeros((bmax, world, 32, 2), dtype=torch.float32, device=self.device)
            self.ws = torch.empty(bmax * 512 * 64, dtype=torch.float32, device=self.device)
            torch.cuda.synchronize()
            self.flags, flag_ptrs = self._shared(world * 4, torch.int32)
            self.slots, slot_ptrs = self._shared(2 * bmax * world * 64 * 4, torch.float32)
        c = _lib.PeerComm()
        c.world, c.rank, c.Bmax = world, rank, bmax
        c.flags, c.seq, c.done, c.cur_stats = self.flags.data_ptr(), self.seq.data_ptr(), self.done.data_ptr(), self.cur_stats.data_ptr()
        for q in range(world):
            c.peer_flags[q] = flag_ptrs[q]
            c.stats_slots[q] = slot_ptrs[q]
        self.c = c
        self._stats_of = None      # data_ptr of the tensor whose statistics cur_stats holds
        # layout switches inside the producing GEMM's epilogue (scatter_plan): "0" off, "1" every supported shape, "aligned" (default) only
        # shapes whose 32-row epilogue patches never straddle a rank's pixel range or a frame (H*W/P and H*W multiples of 32)
        self.fused = os.environ.get("VC_PEER_FUSED", "aligned")
        # ... and only for frame groups of at most this many ranks: 2 is what was validated on hardware (round 2: probe at the real level shapes,
        # sharded forward vs single GPU, graph replay, bench); the kernels handle up to 4 ranks (VC_PEER_FUSED_MAXP=4)
        self.fused_max_p = int(os.environ.get("VC_PEER_FUSED_MAXP", "2"))
        self.fused_switches = 0

    # -- CUDA IPC plumbing (setup only) -------------------------------------------------------------
    class _Raw:
        """__cuda_array_interface__ over a raw device allocation, so torch can alias it."""

        def __init__(self, ptr, nbytes):
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None}

    def _shared(self, nbytes: int, dtype):
        """A zero-filled IPC-shareable allocation of `nbytes` on EVERY rank of the group (collective).  Returns (own tensor of
        `dtype`, [device pointer of rank q's allocation as mapped into this process]); the mapping is opened with this rank's
        compute device current, which is what gives its kernels access over NVLink."""
        import ctypes as C
        from . import _lib
        nbytes = (int(nbytes) + 255) // 256 * 256
        ptr, handle = C.c_void_p(), (C.c_uint8 * 64)()
        _lib.check(self.lib.vc_peer_alloc(nbytes, C.byref(ptr), handle), "vc_peer_alloc")
        self._own_ptrs.append(ptr.value)
        handles = [None] * self.world
        self.dist.all_gather_object(handles, (bytes(handle), torch.cuda.current_device()), group=self.group)
        ptrs = []
        for q, (hb, dev_q) in enumerate(handles):
            if q == self.rank:
                ptrs.append(ptr.value)
                continue
            _lib.check(self.lib.vc_enable_peer_access(int(dev_q)), "vc_enable_peer_access")
            rp = C.c_void_p()
            _lib.check(self.lib.vc_peer_open((C.c_uint8 * 64).from_buffer_copy(hb), C.byref(rp)), "vc_peer_open")
            self._peer_ptrs.append(rp.value)
            ptrs.append(rp.value)
        own = torch.as_tensor(self._Raw(ptr.value, nbytes), device=self.device).view(dtype)
        self.dist.barrier(group=self.group)
        return own, ptrs

    def _buffer(self, name: str, numel: int):
        """fp16 receive buffer `name` with room for `numel` elements on EVERY rank (collective: all ranks grow it together)."""
        ent = self._bufs.get(name)
        if ent is None or ent[2] < numel:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("PeerFrameComm: a receive buffer must grow during CUDA-graph capture; run one eager forward first")
            torch.cuda.synchronize()
            self.dist.barrier(group=self.group)          # nobody still writes into the old mapping
            with torch.cuda.device(self.device):
                own, ptrs = self._shared(numel * 2, torch.float16)
            ent = (own, ptrs, numel)
            self._bufs[name] = ent
        return ent

    def _exchange(self, h: torch.Tensor, B: int, HW: int, to_sites: bool) -> torch.Tensor:
        import ctypes as C
        from . import _lib
        P, Cc = self.world, h.shape[1]
        assert HW % P == 0, f"H*W={HW} must be divisible by the world size {P}"
        assert h.is_contiguous() and h.dtype == torch.float16 and B <= self.bmax
        HWl = HW // P
        Tl = self.ranges[self.rank][1] - self.ranges[self.rank][0]
        tmax = max(f1 - f0 for f0, f1 in self.ranges)
        out_rows = B * self.T * HWl if to_sites else B * Tl * HW
        cap = B * (self.T * HWl if to_sites else tmax * HW) * Cc        # same on every rank
        own, ptrs, _ = self._buffer("sites" if to_sites else "frames", cap)
        dst = (C.c_void_p * P)(*ptrs)
        f0 = (C.c_int32 * (P + 1))(*([r[0] for r in self.ranges] + [self.T]))
        _lib.check(self.lib.vc_peer_exchange(C.byref(self.c), h.data_ptr(), dst, int(to_sites), B, self.T, HW, Cc, f0, int(to_sites),
                                             self.ws.data_ptr(), self.ws.numel() * 4, torch.cuda.current_stream().cuda_stream), "vc_peer_exchange")
        sent = h.numel() * 2
        self.bytes_moved += sent * (P - 1) // P if to_sites else sent - B * Tl * HWl * Cc * 2
        out = own[:out_rows * Cc].view(out_rows, Cc)
        self._stats_of = out.data_ptr() if to_sites else None
        return out

    def _to_sites(self, h: torch.Tensor, B: int, HW: int) -> torch.Tensor:
        return self._exchange(h, B, HW, True)

    def _to_frames(self, t: torch.Tensor, B: int, HW: int) -> torch.Tensor:
        return self._exchange(t, B, HW, False)

    def groupnorm5d(self, x, B, gamma, beta, eps, silu, stat_rows, fresh: bool):
        import ctypes as C
        from . import _lib, ops
        stream = torch.cuda.current_stream().cuda_stream
        rows, Cc = x.shape
        if not (fresh and self._stats_of == x.data_ptr()):
            e0 = self._mark()
            _lib.check(self.lib.vc_peer_groupnorm_stats(C.byref(self.c), x.data_ptr(), Cc, B, rows // B, self.ws.data_ptr(), self.ws.numel() * 4,
                                                        stream), "vc_peer_groupnorm_stats")
            self._done(e0)
        self._stats_of = None
        out = torch.empty_like(x)
        _lib.check(self.lib.vc_groupnorm_apply_parts(x.data_ptr(), Cc, B, rows // B, self.cur_stats.data_ptr(), self.world, stat_rows,
                                                     gamma.data_ptr(), beta.data_ptr(), eps, int(silu), out.data_ptr(), stream),
                   "vc_groupnorm_apply_parts")
        return out

    # -- layout switch fused into the producing GEMM's epilogue ------------------------------------------------
    def scatter_plan(self, to_sites: bool, B: int, HW: int, Cc: int):
        """A plan for ops.conv3x3 / conv_temporal / linear(peer=plan): the GEMM that PRODUCES the tensor stores its output tiles straight
        into the receive buffers of the ranks that own them in the other layout (TMA stores over NVLink, overlapped with its MMAs), and
        a one-CTA kernel completes the switch (rendezvous + the cross-rank GroupNorm sums from the GEMM's own partial sums).  Replaces
        GEMM -> local tensor -> peer_exchange_kernel.  None when the shape is not supported (the caller then switches separately)."""
        P = self.world
        if self.fused == "0" or P > min(4, self.fused_max_p) or HW % P != 0 or Cc % 32 != 0 or B > self.bmax:
            return None
        if self.fused == "aligned" and ((HW // P) % 32 != 0 or HW % 32 != 0):
            return None
        # the decision must be the same on every rank of the group: it depends on ALL frame ranges, not on this rank's
        for f0, f1 in self.ranges:
            if f1 - f0 == 0 or (B > 1 and ((f1 - f0) * HW) % 128 != 0):
                return None
        return _ScatterPlan(self, to_sites, B, HW, Cc)

    def owns(self, t: torch.Tensor) -> bool:
        """True if `t` is a view of one of the reusable receive buffers."""
        p = t.data_ptr()
        return any(ent[0].data_ptr() <= p < ent[0].data_ptr() + ent[0].numel() * 2 for ent in self._bufs.values())

    def close(self):
        """Unmap the peers' buffers and free the own ones (call on every rank after a barrier; optional at process exit)."""
        for p in self._peer_ptrs:
            self.lib.vc_peer_close(p)
        for p in self._own_ptrs:
            self.lib.vc_peer_free(p)
        self._peer_ptrs, self._own_ptrs, self._bufs = [], [], {}


class _ScatterPlan:
    """One fused layout switch (PeerFrameComm.scatter_plan): attach() fills the GEMM descriptor, finish() completes the switch."""

    def __init__(self, comm: "PeerFrameComm", to_sites: bool, B: int, HW: int, Cc: int):
        from . import _lib
        self.comm, self.to_sites, self.B, self.HW, self.C = comm, to_sites, B, HW, Cc
        P = comm.world
        HWl = HW // P
        Tl = comm.ranges[comm.rank][1] - comm.ranges[comm.rank][0]
        tmax = max(f1 - f0 for f0, f1 in comm.ranges)
        self.rows_in = B * Tl * HW if to_sites else B * comm.T * HWl
        self.rows_out = B * comm.T * HWl if to_sites else B * Tl * HW
        cap = B * (comm.T * HWl if to_sites else tmax * HW) * Cc            # same on every rank (as in _exchange)
        self.own, ptrs, _ = comm._buffer("sites" if to_sites else "frames", cap)
        g = _lib.GemmPeer()
        g.mode, g.world, g.rank, g.B, g.T, g.HW = (1 if to_sites else 2), P, comm.rank, B, comm.T, HW
        for q in range(P):
            g.f0[q] = comm.ranges[q][0]
            g.dst[q] = ptrs[q]
        g.f0[P] = comm.T
        self.g = g

    def attach(self, d):
        """Route the output of the GEMM described by `d` (its `out` must not be set by the caller)."""
        import ctypes as C
        d.peer = C.addressof(self.g)
        d.out, d.ldo = self.own.data_ptr(), self.C            # never written: the epilogue stores through the per-rank maps

    def finish(self, gn_part):
        """Rendezvous (+ cross-rank GroupNorm sums for frames -> sites).  Returns the switched tensor (a view of the receive buffer)."""
        import ctypes as C
        from . import _lib
        comm = self.comm
        geom = None
        if self.to_sites and gn_part is not None:
            Tl = comm.ranges[comm.rank][1] - comm.ranges[comm.rank][0]
            geom = gn_part.geom(self.B, Tl * self.HW)
        # geom None (channel counts whose GroupNorm groups are not multiples of the 10-channel sub-groups, e.g. reduced test widths):
        # rendezvous only; groupnorm5d() then takes its statistics with a pass over the received tensor (vc_peer_groupnorm_stats)
        e0 = comm._mark()
        _lib.check(comm.lib.vc_peer_finish_scatter(C.byref(comm.c), C.byref(geom) if geom is not None else None, self.C, self.B, comm.ws.data_ptr(),
                                                   comm.ws.numel() * 4, torch.cuda.current_stream().cuda_stream), "vc_peer_finish_scatter")
        comm._done(e0)
        P = comm.world
        sent = self.rows_in * self.C * 2
        Tl = comm.ranges[comm.rank][1] - comm.ranges[comm.rank][0]
        comm.bytes_moved += sent * (P - 1) // P if self.to_sites else sent - self.B * Tl * (self.HW // P) * self.C * 2
        comm.fused_switches += 1
        out = self.own[:self.rows_out * self.C].view(self.rows_out, self.C)
        comm._stats_of = out.data_ptr() if geom is not None else None
        return out


class CfgComm:
    """Classifier-free-guidance split: the conditional and unconditional U-Net forwards of a DDIM step are independent
    (ddim.py:223-224), so the first half of the ranks computes `cond`, the second half `uncond`, and rank i swaps its
    3.7 MB prediction with rank i + world/2 through a 2-rank all-gather."""

    def __init__(self, dist, branch: int, pair_group):
        self.dist, self.branch, self.pair_group = dist, branch, pair_group

    def exchange(self, v_mine: torch.Tensor):
        buf = v_mine.new_empty((2, *v_mine.shape))
        self.dist.all_gather_into_tensor(buf.view(-1), v_mine.contiguous().view(-1), group=self.pair_group)   # pair group rank order = (cond, uncond)
        return buf[0], buf[1]

    def exchange3(self, v_a: torch.Tensor, v_b: torch.Tensor = None):
        """Three-way guidance: branch 0 passes (v_cond, v_img), branch 1 passes v_uncond (its second slot is padding); one all-gather
        of a 2-slot buffer per pair.  Returns (v_cond, v_uncond, v_img) on every rank."""
        mine = v_a.new_zeros((2, *v_a.shape))
        mine[0] = v_a
        if v_b is not None:
            mine[1] = v_b
        buf = v_a.new_empty((2, 2, *v_a.shape))
        self.dist.all_gather_into_tensor(buf.view(-1), mine.view(-1), group=self.pair_group)
        return buf[0, 0], buf[1, 0], buf[0, 1]


def _make_comm(dist, rank, world, group, device, peer: bool):
    if peer and world > 1 and device is not None and torch.device(device).type == "cuda":
        comm, err = None, None
        try:
            comm = PeerFrameComm(dist, rank, world, group, device)
        except Exception as e:                       # e.g. CUDA IPC not permitted in this container
            err = e
        ok = torch.tensor([0.0 if comm is None else 1.0], device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)      # all ranks of the group take the same path
        if float(ok) > 0:
            return comm
        import warnings
        warnings.warn(f"viewcrafter_b200.parallel: NVLink peer-memory exchange unavailable ({err!r}); using the NCCL collectives")
    return FrameComm(dist, rank, world, group)


def shard_model(model, dist, rank: int, world: int, cfg_split: bool = True, peer: bool = None):
    """Distribute the denoise step over `world` ranks (weights stay replicated: 2.9 GB fp16 per GPU).

    world even and cfg_split: 2-way CFG split x (world/2)-way frame sharding -- e.g. 8 GPUs = 2 x 4 with frames 7/6/6/6
    (ideal 7.1x) instead of 8-way frames 4/3x7 (ideal 6.25x).  Otherwise pure frame sharding.
    Every rank must call this (it creates process groups collectively).  Returns the FrameComm (or None).

    A model with a ``first_stage_model`` also gets ``model._vae``: a FrameComm over the whole world, which makes
    ``synthesis.get_latent_z`` and the decode of ``synthesis.image_guided_synthesis`` split their per-frame VAE work over all
    ranks (vae_encode_sharded / vae_decode_sharded)."""
    if world > 1 and getattr(model, "first_stage_model", None) is not None:
        model._vae = FrameComm(dist, rank, world, None)          # the VAE has no CFG branches: all ranks share its frames
    unet = model.model.diffusion_model if hasattr(model, "model") else model
    try:
        device = next(unet.parameters()).device
    except StopIteration:
        device = None
    if peer is None:           # NVLink peer-memory kernels on CUDA (VC_PEER_COMM=0: NCCL collectives); the CPU double uses gloo
        import os
        peer = os.environ.get("VC_PEER_COMM", "1") != "0"
    if cfg_split and world % 2 == 0 and hasattr(model, "model"):
        P = world // 2
        frame_groups = [dist.new_group(list(range(b * P, (b + 1) * P))) for b in range(2)]
        pair_groups = [dist.new_group([i, i + P]) for i in range(P)]
        branch, r = rank // P, rank % P
        model._cfg = CfgComm(dist, branch, pair_groups[r])
        unet._comm = _make_comm(dist, r, P, frame_groups[branch], device, peer) if P > 1 else None
        return unet._comm
    unet._comm = _make_comm(dist, rank, world, None, device, peer)
    return unet._comm


# -- the VAE stages of a clip ------------------------------------------------------------------------------------------------------
# The VAE works on one frame at a time (per-frame GroupNorm, one single-image AttnBlock per frame), so its work splits by frame with
# no communication inside it: rank r runs its frame range of every sample, then the results are all-gathered (FrameComm.gather_frames).
# Only attributes the reference's VIPLatentDiffusion also has are used (first_stage_model.encode, get_first_stage_encoding,
# decode_first_stage, perframe_ae), so the reference model with the viewcrafter_b200 networks swapped in is sharded the same way.

def vae_encode_sharded(model, videos: torch.Tensor) -> torch.Tensor:
    """videos [b, c, T, H, W] -> latents [b, c', T, H/8, W/8] on every rank, equal to what get_latent_z returns in one process.

    Rank r encodes frames [t0, t1) of every sample (one call per frame when perframe_ae, else one call) and keeps the posterior
    moments; the moments are all-gathered, and every rank then draws the posterior samples itself in the reference's order
    (ddpm3d.py:620-644: one draw per frame in (b t) order when perframe_ae, else one draw over all frames).  So every rank consumes
    the CPU generator exactly as a single process does and ends in its state: x_T, the per-step noise and the next clip's draws
    stay the reference's.  (Calling encode_first_stage on a frame slice would draw the noise of the wrong frames.)"""
    from .distributions import posterior_class
    comm = model._vae
    b, c, T, H, W = videos.shape
    t0, t1 = comm.bind(T)
    vae = model.first_stage_model
    if t1 > t0:
        x = videos[:, :, t0:t1].permute(0, 2, 1, 3, 4).reshape(b * (t1 - t0), c, H, W)
        posts = [vae.encode(x[i:i + 1]) for i in range(x.shape[0])] if model.perframe_ae else [vae.encode(x)]
        cls = type(posts[0])                        # the reference's own posterior class when its AutoencoderKL is used
        m = torch.cat([p.parameters for p in posts], 0)
        local = m.reshape(b, t1 - t0, *m.shape[1:]).permute(0, 2, 1, 3, 4)
    else:
        # T < world: no frames here, only the gather padding.  The fp32 moments and the posterior class are what
        # viewcrafter_b200's AutoencoderKL.encode returns (posterior_class() subclasses the reference's class when that is loaded).
        f = 2 ** (len(vae.encoder.down) - 1)
        local = videos.new_empty((b, 2 * vae.embed_dim, 0, H // f, W // f), dtype=torch.float32)
        cls = posterior_class()
    moments = comm.gather_frames(local, T).permute(0, 2, 1, 3, 4).flatten(0, 1)      # [(b T), 2*embed, h, w]
    if model.perframe_ae:
        z = torch.cat([model.get_first_stage_encoding(cls(moments[i:i + 1])).detach() for i in range(b * T)], 0)
    else:
        z = model.get_first_stage_encoding(cls(moments)).detach()
    return z.reshape(b, T, *z.shape[1:]).permute(0, 2, 1, 3, 4)


def vae_decode_sharded(model, samples: torch.Tensor) -> torch.Tensor:
    """latents [b, c, T, h, w] -> the decoded video [b, out_ch, T, 8h, 8w] on every rank: rank r decodes frames [t0, t1) through
    the model's own decode_first_stage (so its perframe_ae / decode_batch rules apply to the slice), then the frames are gathered."""
    comm = model._vae
    b, _, T, h, w = samples.shape
    t0, t1 = comm.bind(T)
    if t1 > t0:
        local = model.decode_first_stage(samples[:, :, t0:t1])
    else:                                                                      # T < world: only the gather padding
        dec = model.first_stage_model.decoder
        f = 2 ** (len(dec.up) - 1)
        local = samples.new_empty((b, dec.conv_out.out_channels, 0, h * f, w * f))
    return comm.gather_frames(local, T)
