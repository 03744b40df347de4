"""Drop-in ``UNetModel`` (reference: lvdm/modules/networks/openaimodel3d.py:281-603).

Same constructor kwargs, same ``forward(x, timesteps, context, features_adapter, fs, **kw)`` and the same
state-dict keys/shapes (SURVEY.md Appendix B) so the reference checkpoint loads with ``strict=True``.  The
``torch.nn`` modules below are *parameter holders only*: ``forward`` never calls them.  All arithmetic runs in
libvc_b200.so on channels-last fp16 activations (``rows = (b t) h w``, columns = channels):

    ResBlock            -> GroupNorm+SiLU kernel, 9-tap tcgen05 GEMM (+emb bias), again, 1x1 skip GEMM fused as
                           residual, then 4x [5-D GroupNorm+SiLU, 3-tap temporal GEMM]          (:210-279)
    SpatialTransformer  -> GroupNorm, proj_in GEMM, LN, fused-QKV GEMM, tcgen05 flash attention, out-proj GEMM
                           (+res), LN, q GEMM, text + image cross attention (accumulate), LN, GEGLU GEMM, FF GEMM,
                           proj_out GEMM (+x_in)                                                  (attention.py:249-310)
    TemporalTransformer -> same with the temporal (T<=32) attention kernel, no transposes: tokens stay in
                           (t, h, w) row order and the kernel strides over t                      (attention.py:313-412)
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
import torch.nn as nn

from . import ops


def _zero(m: nn.Module) -> nn.Module:
    for p in m.parameters():
        nn.init.zeros_(p)
    return m


_LN_FOLD = os.environ.get("VC_LN_FOLD", "1") != "0"   # fold norm1/2/3 into their consumer GEMMs (A/B switch, read at import)


def _ln_linear(Q: dict, x: torch.Tensor, name: str, ln: str, st=None, **kw) -> torch.Tensor:
    """LayerNorm -> Linear of a transformer block: folded (row statistics + GEMM epilogue) or as two passes.  `st`: the (mean, rstd)
    of x if the GEMM that produced x already gathered them (ops.linear(..., ln_out=True)); otherwise a statistics pass reads x."""
    if Q[name + "_cs"] is not None:
        return ops.linear(x, Q[name], bias=Q[name + "_b"], ln=(st if st is not None else ops.layernorm_stats(x), Q[name + "_cs"]), **kw)
    return ops.linear(ops.layernorm(x, *Q[ln]), Q[name], bias=Q[name + "_b"], **kw)


# cfg_shared_prefix=True asks for the shared CFG prefix on one GPU only: the two-way sampler sends it to frame-sharded forwards too, which
# run the plain B=2 path.  This value asks for it under frame sharding as well (the three-way sampler's stacked calls).
SHARED_PREFIX_ANY_LAYOUT = "any_layout"


def _unsupported(flag: str):
    raise NotImplementedError(f"viewcrafter_b200.UNetModel: option {flag} is not on the ViewCrafter inference path")


# --------------------------------------------------------------------------------------------------
# parameter holders (names are load-bearing, incl. the upstream 'temopral_conv' spelling)
# --------------------------------------------------------------------------------------------------
class _Attn(nn.Module):
    def __init__(self, dim: int, ctx_dim: Optional[int], heads: int, image_branch: bool):
        super().__init__()
        inner = heads * 64
        kd = ctx_dim or dim
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_k = nn.Linear(kd, inner, bias=False)
        self.to_v = nn.Linear(kd, inner, bias=False)
        self.to_out = nn.Sequential(nn.Linear(inner, dim), nn.Dropout(0.0))
        if image_branch:
            self.to_k_ip = nn.Linear(kd, inner, bias=False)
            self.to_v_ip = nn.Linear(kd, inner, bias=False)


class _GEGLU(nn.Module):
    def __init__(self, dim, inner):
        super().__init__()
        self.proj = nn.Linear(dim, inner * 2)


class _FF(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.net = nn.Sequential(_GEGLU(dim, dim * 4), nn.Dropout(0.0), nn.Linear(dim * 4, dim))


class _TBlock(nn.Module):
    def __init__(self, dim, heads, ctx_dim, image_branch):
        super().__init__()
        self.attn1 = _Attn(dim, None, heads, False)
        self.ff = _FF(dim)
        self.attn2 = _Attn(dim, ctx_dim, heads, image_branch)
        self.norm1, self.norm2, self.norm3 = nn.LayerNorm(dim), nn.LayerNorm(dim), nn.LayerNorm(dim)


class _Transformer(nn.Module):
    """kind 'S' (SpatialTransformer) or 'T' (TemporalTransformer); conv1d=True gives init_attn's Conv1d projections."""

    def __init__(self, kind, channels, heads, depth, ctx_dim, image_branch, conv1d=False):
        super().__init__()
        self.kind, self.channels, self.heads = kind, channels, heads
        inner = heads * 64
        self.norm = nn.GroupNorm(32, channels, eps=1e-6, affine=True)
        mk = (lambda i, o: nn.Conv1d(i, o, 1)) if conv1d else nn.Linear
        self.proj_in = mk(channels, inner)
        self.transformer_blocks = nn.ModuleList([
            _TBlock(inner, heads, ctx_dim if kind == "S" else None, image_branch and kind == "S") for _ in range(depth)])
        self.proj_out = _zero(mk(inner, channels))


class _TemporalConv(nn.Module):
    def __init__(self, c):
        super().__init__()
        conv = lambda: nn.Conv3d(c, c, (3, 1, 1), padding=(1, 0, 0))
        self.conv1 = nn.Sequential(nn.GroupNorm(32, c), nn.SiLU(), conv())
        self.conv2 = nn.Sequential(nn.GroupNorm(32, c), nn.SiLU(), nn.Dropout(0.0), conv())
        self.conv3 = nn.Sequential(nn.GroupNorm(32, c), nn.SiLU(), nn.Dropout(0.0), conv())
        self.conv4 = nn.Sequential(nn.GroupNorm(32, c), nn.SiLU(), nn.Dropout(0.0), _zero(conv()))


class _Res(nn.Module):
    def __init__(self, cin, emb_ch, cout, temporal):
        super().__init__()
        self.cin, self.cout = cin, cout
        self.in_layers = nn.Sequential(nn.GroupNorm(32, cin), nn.SiLU(), nn.Conv2d(cin, cout, 3, padding=1))
        self.emb_layers = nn.Sequential(nn.SiLU(), nn.Linear(emb_ch, cout))
        self.out_layers = nn.Sequential(nn.GroupNorm(32, cout), nn.SiLU(), nn.Dropout(0.0),
                                        _zero(nn.Conv2d(cout, cout, 3, padding=1)))
        self.skip_connection = nn.Identity() if cin == cout else nn.Conv2d(cin, cout, 1)
        if temporal:
            self.temopral_conv = _TemporalConv(cout)


class _Down(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.op = nn.Conv2d(c, c, 3, stride=2, padding=1)


class _Up(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, padding=1)


class _Stage(nn.Sequential):
    pass


# --------------------------------------------------------------------------------------------------
class UNetModel(nn.Module):
    def __init__(self, in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions, dropout=0.0,
                 channel_mult=(1, 2, 4, 8), conv_resample=True, dims=2, context_dim=None, use_scale_shift_norm=False,
                 resblock_updown=False, num_heads=-1, num_head_channels=-1, transformer_depth=1, use_linear=False,
                 use_checkpoint=False, temporal_conv=False, tempspatial_aware=False, temporal_attention=True,
                 use_relative_position=True, use_causal_attention=False, temporal_length=None, use_fp16=False,
                 addition_attention=False, temporal_selfatt_only=True, image_cross_attention=False,
                 image_cross_attention_scale_learnable=False, default_fs=4, fs_condition=False):
        super().__init__()
        if num_head_channels != 64:
            _unsupported("num_head_channels != 64 (the attention kernels are specialised for head_dim 64)")
        for bad, name in ((use_scale_shift_norm, "use_scale_shift_norm"), (resblock_updown, "resblock_updown"),
                          (tempspatial_aware, "tempspatial_aware"), (use_relative_position, "use_relative_position"),
                          (use_causal_attention, "use_causal_attention"), (not use_linear, "use_linear=False"),
                          (not conv_resample, "conv_resample=False"), (dims != 2, "dims != 2"),
                          (not temporal_selfatt_only, "temporal_selfatt_only=False"),
                          (image_cross_attention_scale_learnable, "image_cross_attention_scale_learnable")):
            if bad:
                _unsupported(name)
        self.in_channels, self.model_channels, self.out_channels = in_channels, model_channels, out_channels
        self.num_res_blocks, self.attention_resolutions, self.channel_mult = num_res_blocks, attention_resolutions, channel_mult
        self.dropout, self.use_checkpoint = dropout, use_checkpoint
        self.temporal_attention, self.temporal_length = temporal_attention, temporal_length
        self.addition_attention, self.image_cross_attention = addition_attention, image_cross_attention
        self.default_fs, self.fs_condition = default_fs, fs_condition
        self.dtype = torch.float16 if use_fp16 else torch.float32
        mc, ted = model_channels, model_channels * 4

        mlp = lambda: nn.Sequential(nn.Linear(mc, ted), nn.SiLU(), nn.Linear(ted, ted))
        self.time_embed = mlp()
        if fs_condition:
            self.fps_embedding = mlp()
            _zero(self.fps_embedding[-1])

        def attn_layers(ch):
            heads = ch // 64
            layers = [_Transformer("S", ch, heads, transformer_depth, context_dim, image_cross_attention)]
            if temporal_attention:
                layers.append(_Transformer("T", ch, heads, transformer_depth, None, False))
            return layers

        self.input_blocks = nn.ModuleList([_Stage(nn.Conv2d(in_channels, mc, 3, padding=1))])
        if addition_attention:
            self.init_attn = _Stage(_Transformer("T", mc, 8, transformer_depth, None, False, conv1d=True))
        skip_ch, ch, ds = [mc], mc, 1
        for level, mult in enumerate(channel_mult):
            for _ in range(num_res_blocks):
                layers: List[nn.Module] = [_Res(ch, ted, mult * mc, temporal_conv)]
                ch = mult * mc
                if ds in attention_resolutions:
                    layers += attn_layers(ch)
                self.input_blocks.append(_Stage(*layers))
                skip_ch.append(ch)
            if level != len(channel_mult) - 1:
                self.input_blocks.append(_Stage(_Down(ch)))
                skip_ch.append(ch)
                ds *= 2
        mid: List[nn.Module] = [_Res(ch, ted, ch, temporal_conv),
                                _Transformer("S", ch, ch // 64, transformer_depth, context_dim, image_cross_attention)]
        if temporal_attention:
            mid.append(_Transformer("T", ch, ch // 64, transformer_depth, None, False))
        mid.append(_Res(ch, ted, ch, temporal_conv))
        self.middle_block = _Stage(*mid)
        self.output_blocks = nn.ModuleList()
        for level, mult in list(enumerate(channel_mult))[::-1]:
            for i in range(num_res_blocks + 1):
                layers = [_Res(ch + skip_ch.pop(), ted, mult * mc, temporal_conv)]
                ch = mult * mc
                if ds in attention_resolutions:
                    layers += attn_layers(ch)
                if level and i == num_res_blocks:
                    layers.append(_Up(ch))
                    ds //= 2
                self.output_blocks.append(_Stage(*layers))
        self.out = nn.Sequential(nn.GroupNorm(32, ch), nn.SiLU(), _zero(nn.Conv2d(mc, out_channels, 3, padding=1)))

        self._packed = None
        self._kv_caches = []        # cross-attention K/V projections of the last three contexts (see _kv_projector)
        self._canon = []            # [ref, version, private snapshot] of the last three contexts (see _canonical_context)
        self._kv_cache = {}
        self._comm = None           # set by viewcrafter_b200.parallel.shard_model for frame-sharded multi-GPU execution
        self._graph_mode = os.environ.get("VC_UNET_GRAPH", "0") == "1"     # see enable_cuda_graph
        self._graphs = {}
        self.graph_replayed_launches = 0    # kernels of this library executed through graph replays (bench.py's gpu_launches)
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.invalidate_packed())

    # ------------------------------------------------------------------------------------------
    # weight packing: fp32 checkpoint tensors -> kernel layouts (fp16 K-major GEMM operands, fp32 norm/bias)
    # ------------------------------------------------------------------------------------------
    def invalidate_packed(self):
        self._packed = None
        self._kv_caches, self._kv_cache, self._canon = [], {}, []
        self._graphs = {}

    def enable_cuda_graph(self, on: bool = True):
        """Replay the whole forward as ONE CUDA graph (SURVEY.md 8 f2 / 8b): the denoise loop calls forward ~100 times per
        clip with the same shapes, the same context tensor and the same weights, so the ~1000 kernel launches (and their
        host-side tensor-map encodes) of a forward are captured on the second call with a given (shape, context) and replayed
        afterwards: per call the host does two small input copies and one graph launch.  Results are those of the eager path
        (same kernels, same order).  Off by default; bench.py / synthesis.py switch it on.  A new context tensor, an in-place
        write to it, a new shape or new weights lead to a new capture; at most 4 graphs are kept."""
        self._graph_mode = bool(on)
        if not on:
            self._graphs = {}
        return self

    def _apply(self, fn, *a, **k):
        # a pure device move (.cuda() / .to(device)) carries the packed kernel operands along (H2D copies, no repacking);
        # anything that changes dtypes drops them
        packed = self._packed if ops.is_device_only(fn) else None
        self._packed = None
        self._kv_caches, self._kv_cache, self._canon = [], {}, []
        self._graphs = {}
        r = super()._apply(fn, *a, **k)
        if packed is not None:
            self._packed = ops.tree_apply(packed, fn)
            self._packed["device"] = self.time_embed[0].weight.device
        return r

    @staticmethod
    def _f32(t):
        return t.detach().float().contiguous()

    def _pack_res(self, m: _Res):
        f = self._f32
        P = dict(kind="R", cin=m.cin, cout=m.cout)
        P["gn1"] = (f(m.in_layers[0].weight), f(m.in_layers[0].bias))
        P["w1"] = ops.pack_conv3x3(m.in_layers[2].weight.detach())
        P["emb_w"] = f(m.emb_layers[1].weight)
        P["emb_b"] = f(m.emb_layers[1].bias + m.in_layers[2].bias)       # conv1 bias folded into the per-batch emb row
        P["gn2"] = (f(m.out_layers[0].weight), f(m.out_layers[0].bias))
        P["w2"] = ops.pack_conv3x3(m.out_layers[3].weight.detach())
        P["b2"] = f(m.out_layers[3].bias)
        if isinstance(m.skip_connection, nn.Conv2d):
            P["skip_w"] = ops.pack_linear(m.skip_connection.weight.detach())
            P["skip_b"] = f(m.skip_connection.bias)
        if hasattr(m, "temopral_conv"):
            tc = m.temopral_conv
            P["tconv"] = [(f(seq[0].weight), f(seq[0].bias), ops.pack_conv_temporal(seq[-1].weight.detach()), f(seq[-1].bias))
                          for seq in (tc.conv1, tc.conv2, tc.conv3, tc.conv4)]
        return P

    def _pack_tf(self, m: _Transformer):
        f = self._f32
        P = dict(kind=m.kind, heads=m.heads, C=m.channels)
        P["gn"] = (f(m.norm.weight), f(m.norm.bias))
        P["in_w"], P["in_b"] = ops.pack_linear(m.proj_in.weight.detach()), f(m.proj_in.bias)
        P["out_w"], P["out_b"] = ops.pack_linear(m.proj_out.weight.detach()), f(m.proj_out.bias)
        blocks = []
        for b in m.transformer_blocks:
            Q = {}
            # norm1/2/3 feed exactly one linear each (attention.py:283-292): fold them into it -- the GEMM reads the raw
            # residual stream and its epilogue applies (mean, rstd); LayerNorm shrinks to a read-only statistics pass.
            # VC_LN_FOLD=0 keeps the separate LayerNorm pass (A/B switch).
            n1, n2, n3 = ((ln.weight.detach(), ln.bias.detach()) for ln in (b.norm1, b.norm2, b.norm3))
            a1, a2 = b.attn1, b.attn2
            cat = lambda *ws: torch.cat(ws, 0).detach()
            if _LN_FOLD:
                fold = ops.fold_layernorm
            else:
                fold = lambda w, g, bta: (ops.pack_linear(w), None, None)
                Q["ln1"], Q["ln2"], Q["ln3"] = ((f(g), f(bta)) for g, bta in (n1, n2, n3))
            Q["qkv1"], Q["qkv1_cs"], Q["qkv1_b"] = fold(cat(a1.to_q.weight, a1.to_k.weight, a1.to_v.weight), *n1)
            Q["o1_w"], Q["o1_b"] = ops.pack_linear(a1.to_out[0].weight.detach()), f(a1.to_out[0].bias)
            if m.kind == "T":
                Q["qkv2"], Q["qkv2_cs"], Q["qkv2_b"] = fold(cat(a2.to_q.weight, a2.to_k.weight, a2.to_v.weight), *n2)
            else:
                Q["q2"], Q["q2_cs"], Q["q2_b"] = fold(a2.to_q.weight.detach(), *n2)
                Q["kv_txt"] = torch.cat([a2.to_k.weight, a2.to_v.weight], 0).detach().to(torch.float16).contiguous()
                if hasattr(a2, "to_k_ip"):
                    Q["kv_img"] = torch.cat([a2.to_k_ip.weight, a2.to_v_ip.weight], 0).detach().to(torch.float16).contiguous()
            Q["o2_w"], Q["o2_b"] = ops.pack_linear(a2.to_out[0].weight.detach()), f(a2.to_out[0].bias)
            if _LN_FOLD:
                Q["ff1"], Q["ff1_b"], Q["ff1_cs"] = ops.pack_geglu_ln(b.ff.net[0].proj.weight.detach(), b.ff.net[0].proj.bias.detach(), *n3)
            else:
                Q["ff1"], Q["ff1_b"] = ops.pack_geglu(b.ff.net[0].proj.weight.detach(), b.ff.net[0].proj.bias.detach())
                Q["ff1_cs"] = None
            Q["ff2_w"], Q["ff2_b"] = ops.pack_linear(b.ff.net[2].weight.detach()), f(b.ff.net[2].bias)
            blocks.append(Q)
        P["blocks"] = blocks
        return P

    def _pack_stage(self, stage: nn.Sequential):
        f = self._f32
        out = []
        for m in stage:
            if isinstance(m, _Res):
                out.append(self._pack_res(m))
            elif isinstance(m, _Transformer):
                out.append(self._pack_tf(m))
            elif isinstance(m, _Down):
                w = m.op.weight.detach()
                out.append(dict(kind="D", w=w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).to(torch.float16).contiguous(), b=f(m.op.bias)))
            elif isinstance(m, _Up):
                out.append(dict(kind="U", w=ops.pack_upconv3x3(m.conv.weight.detach()), b=f(m.conv.bias)))
            elif isinstance(m, nn.Conv2d):
                out.append(dict(kind="C", w=ops.pack_conv3x3(m.weight.detach(), k_pad=8), b=f(m.bias), cin=m.in_channels))
            else:
                raise TypeError(type(m))
        return out

    def _pack(self):
        f = self._f32
        dev = self.time_embed[0].weight.device          # packing is plain tensor math: it may run before the move to the GPU
        P = dict(device=dev)
        P["time"] = [f(self.time_embed[0].weight), f(self.time_embed[0].bias), f(self.time_embed[2].weight), f(self.time_embed[2].bias)]
        if self.fs_condition:
            P["fps"] = [f(self.fps_embedding[0].weight), f(self.fps_embedding[0].bias), f(self.fps_embedding[2].weight), f(self.fps_embedding[2].bias)]
        P["input"] = [self._pack_stage(s) for s in self.input_blocks]
        if self.addition_attention:
            P["init_attn"] = self._pack_stage(self.init_attn)
        P["middle"] = self._pack_stage(self.middle_block)
        P["output"] = [self._pack_stage(s) for s in self.output_blocks]
        P["out_gn"] = (f(self.out[0].weight), f(self.out[0].bias))
        P["out_w"], P["out_b"] = ops.pack_conv3x3(self.out[2].weight.detach()), f(self.out[2].bias)
        self._packed = P
        return P

    # ------------------------------------------------------------------------------------------
    # block executors (operate on row matrices)
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _res(P, h, skip, emb, B, T, H, W, comm=None):
        BT, HW = B * T, H * W
        a = ops.groupnorm(h, BT, *P["gn1"], 1e-5, True, x2=skip)
        bias1 = ops.small_linear(emb, P["emb_w"], P["emb_b"], silu_in=True)            # [B, Cout] = emb_layers + conv1 bias
        h1 = ops.conv3x3(a, BT, H, W, P["w1"], bias=bias1, bias_z_div=T, gn_out=True)      # gn_out: the epilogue leaves the GroupNorm sums of its output
        b = ops.groupnorm(h1, BT, *P["gn2"], 1e-5, True)
        if "skip_w" in P:
            xs = ops.linear(h, P["skip_w"], bias=P["skip_b"], x2=skip)
        else:
            xs = h
        # multi-GPU: the frames -> sites switch the TemporalConvBlock needs is performed by conv2's own epilogue when the peer-memory path
        # offers a plan (its output tiles go straight to the owning ranks), and the switch back by the last temporal conv's
        to_s = comm.scatter_plan(True, B, HW, P["w2"].shape[0] // 9) if (comm and "tconv" in P) else None
        h2 = ops.conv3x3(b, BT, H, W, P["w2"], bias=P["b2"], res=xs, gn_out=True, peer=to_s)
        if "tconv" in P:
            # TemporalConvBlock: needs every frame of a pixel -> (optionally) transpose frames<->sites across GPUs
            t = ident = h2 if to_s is not None else (comm.to_sites(h2, B, HW) if comm else h2)
            Tg, HWl = (comm.T, HW // comm.world) if comm else (T, HW)
            n_tc, to_f = len(P["tconv"]), None
            for i, (g, be, w3, b3) in enumerate(P["tconv"]):
                t = UNetModel._gn5d(t, B, g, be, 1e-5, True, comm, Tg * HW, fresh=(i == 0))   # statistics over (C/32, T, H, W)
                last = i == n_tc - 1
                to_f = comm.scatter_plan(False, B, HW, w3.shape[0] // 3) if (comm and last) else None
                t = ops.conv_temporal(t, B, Tg, HWl, w3, bias=b3, res=ident if last else None, gn_out=comm is None, peer=to_f)
            h2 = t if to_f is not None else (comm.to_frames(t, B, HW) if comm else t)
        return h2

    @staticmethod
    def _gn5d(x, B, gamma, beta, eps, silu, comm, stat_rows, fresh=False):
        """GroupNorm whose statistics span all frames (and, when sharded, all GPUs: [B,32,2] partial sums are exchanged --
        riding on the layout switch when `fresh`, i.e. x is what comm.to_sites() just returned)."""
        if not comm:
            return ops.groupnorm(x, B, gamma, beta, eps, silu)
        return comm.groupnorm5d(x, B, gamma, beta, eps, silu, stat_rows, fresh)

    @staticmethod
    def _spatial_tf(P, h, ctx, B, T, H, W, expand=False, out_plan=None):
        """expand=True (shared CFG prefix, SURVEY.md App. C.2): `h` holds ONE batch element that is identical for the B (2 or 3)
        guidance branches; everything up to and including attn1 of the first block does not see the context, so it runs once
        and is replicated to B rows right before the first cross-attention."""
        Bc = 1 if expand else B
        BT, HW, heads = Bc * T, H * W, P["heads"]
        C = heads * 64
        fold = _LN_FOLD
        x = ops.linear(ops.groupnorm(h, BT, *P["gn"], 1e-6, False), P["in_w"], bias=P["in_b"], ln_out=fold)
        x, st = x if fold else (x, None)
        for Q in P["blocks"]:
            qkv = _ln_linear(Q, x, "qkv1", "ln1", st)
            a = ops.flash_attn(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], BT, HW, HW, heads)
            x = ops.linear(a, Q["o1_w"], bias=Q["o1_b"], res=x, ln_out=fold)
            x, st = x if fold else (x, None)
            if expand:
                x, h = torch.cat([x] * B, 0), torch.cat([h] * B, 0)
                st = torch.cat([st] * B, 0) if st is not None else None
                expand, Bc, BT = False, B, B * T
            q = _ln_linear(Q, x, "q2", "ln2", st)
            a = torch.empty_like(q)
            for b in range(Bc):
                rows = slice(b * T * HW, (b + 1) * T * HW)
                kv = ctx["kv"](Q, "kv_txt", ctx["text"][b], b)                            # [77, 2C]
                ops.flash_attn(q[rows], kv[:, :C], kv[:, C:], T, HW, kv.shape[0], heads, kv_shared=True, out=a[rows])
                if "kv_img" in Q and ctx["img"] is not None:
                    ki = ctx["kv"](Q, "kv_img", ctx["img"][b], b)                         # [256, 2C] or [T*16, 2C]
                    if ctx["img_per_frame"]:
                        ops.flash_attn(q[rows], ki[:, :C], ki[:, C:], T, HW, ki.shape[0] // T, heads, out=a[rows], accumulate=True)
                    else:
                        ops.flash_attn(q[rows], ki[:, :C], ki[:, C:], T, HW, ki.shape[0], heads, kv_shared=True, out=a[rows], accumulate=True)
            x = ops.linear(a, Q["o2_w"], bias=Q["o2_b"], res=x, ln_out=fold)
            x, st = x if fold else (x, None)
            g = _ln_linear(Q, x, "ff1", "ln3", st, geglu=True)
            last = Q is P["blocks"][-1]
            x = ops.linear(g, Q["ff2_w"], bias=Q["ff2_b"], res=x, ln_out=fold and not last)
            x, st = x if (fold and not last) else (x, None)
        # out_plan (multi-GPU): proj_out's epilogue performs the frames -> sites switch the TemporalTransformer that follows needs
        return ops.linear(x, P["out_w"], bias=P["out_b"], res=h, gn_out=True, peer=out_plan)

    @staticmethod
    def _temporal_tf(P, h, B, T, H, W, comm=None, pre_sites=False):
        """pre_sites: `h` already is in the site layout (the producing GEMM switched it, see _spatial_tf(out_plan=...))."""
        HW, heads = H * W, P["heads"]
        C = heads * 64
        Tg, HWl = (comm.T, HW // comm.world) if comm else (T, HW)
        t_in = h if pre_sites else (comm.to_sites(h, B, HW) if comm else h)
        fold = _LN_FOLD
        x = ops.linear(UNetModel._gn5d(t_in, B, *P["gn"], 1e-6, False, comm, Tg * HW, fresh=True), P["in_w"], bias=P["in_b"], ln_out=fold)
        x, st = x if fold else (x, None)
        for Q in P["blocks"]:
            for ln, wqkv, ow, ob in (("ln1", "qkv1", "o1_w", "o1_b"), ("ln2", "qkv2", "o2_w", "o2_b")):
                qkv = _ln_linear(Q, x, wqkv, ln, st)
                a = torch.empty((qkv.shape[0], C), device=qkv.device, dtype=torch.float16)
                for b in range(B):
                    rows = slice(b * Tg * HWl, (b + 1) * Tg * HWl)
                    ops.temporal_attn(qkv[rows, :C], qkv[rows, C:2 * C], qkv[rows, 2 * C:], Tg, HWl, heads, out=a[rows])
                x = ops.linear(a, Q[ow], bias=Q[ob], res=x, ln_out=fold)
                x, st = x if fold else (x, None)
            g = _ln_linear(Q, x, "ff1", "ln3", st, geglu=True)
            last = Q is P["blocks"][-1]
            x = ops.linear(g, Q["ff2_w"], bias=Q["ff2_b"], res=x, ln_out=fold and not last)
            x, st = x if (fold and not last) else (x, None)
        to_f = comm.scatter_plan(False, B, HW, P["out_w"].shape[0]) if comm else None
        out = ops.linear(x, P["out_w"], bias=P["out_b"], res=t_in, gn_out=comm is None, peer=to_f)
        return out if to_f is not None else (comm.to_frames(out, B, HW) if comm else out)

    def _run_stage(self, stage, h, skip, emb, ctx, B, T, H, W, emb1=None):
        """emb1 (shared CFG prefix): `h` holds ONE batch element common to the B branches; the ResBlock before the first
        SpatialTransformer runs on it with emb1 (the branches' common embedding row) and that transformer expands to B rows."""
        comm, pre_sites = self._comm, False
        Bc = 1 if emb1 is not None else B
        for idx, P in enumerate(stage):
            k = P["kind"]
            if k == "R":
                h = self._res(P, h, skip, emb if Bc == B else emb1, Bc, T, H, W, comm)
                skip = None
            elif k == "S":
                nxt = stage[idx + 1]["kind"] if idx + 1 < len(stage) else None
                plan = comm.scatter_plan(True, B, H * W, P["out_w"].shape[0]) if (comm and nxt == "T") else None
                h = self._spatial_tf(P, h, ctx, B, T, H, W, expand=Bc != B, out_plan=plan)
                Bc = B
                pre_sites = plan is not None
            elif k == "T":
                h = self._temporal_tf(P, h, B, T, H, W, comm, pre_sites=pre_sites)
                pre_sites = False
            elif k == "D":
                cols, H, W = ops.im2col_s2(h, B * T, H, W)
                h = ops.linear(cols, P["w"], bias=P["b"], gn_out=True)
            elif k == "U":
                h = ops.upconv3x3(h, B * T, H, W, P["w"], bias=P["b"])      # upsample folded into four parity sub-convolutions
                H, W = 2 * H, 2 * W
            elif k == "C":
                h = ops.conv3x3(h, B * T, H, W, P["w"], bias=P["b"], gn_out=True)
        return h, H, W

    def _canonical_context(self, context: torch.Tensor) -> torch.Tensor:
        """Map a context tensor to a private, immutable snapshot with the same CONTENT.  The K/V cache and the captured graphs are
        keyed on the snapshot, so they survive callers that rebuild an equal context every step -- the reference's own
        DiffusionWrapper does ``torch.cat(c_crossattn, 1)`` per call (ddpm3d.py:1442).  Fast path: same tensor object with the
        same version counter (no device work).  Otherwise the content is compared with the cached snapshots of the same shape
        (one ``torch.equal`` = one small device->host sync per forward); a genuinely new context is cloned (1.3 MB)."""
        ver = ops.tensor_version(context)
        for ent in self._canon:
            if ent[0] is context and ent[1] == ver and ver is not None:
                return ent[2]
        for i, ent in enumerate(self._canon):
            snap = ent[2]
            if snap.shape == context.shape and snap.dtype == context.dtype and snap.device == context.device and bool(torch.equal(snap, context)):
                ent[0], ent[1] = context, ver
                self._canon.insert(0, self._canon.pop(i))
                return snap
        snap = context.detach().clone()
        self._canon.insert(0, [context, ver, snap])
        for ent in self._canon[3:]:                         # evicted snapshots take their K/V projections and graphs along
            self._kv_caches = [c for c in self._kv_caches if c["ref"] is not ent[2]]
            self._graphs = {k: g for k, g in self._graphs.items() if g["ctx"] is not ent[2]}
        del self._canon[3:]
        return snap

    def _kv_projector(self, context: torch.Tensor, img_range):
        """to_k / to_v (and to_k_ip / to_v_ip) of the cross-attentions see only the context, which a sampling run feeds
        unchanged for all its steps (SURVEY.md App. C.1): project once per (context tensor, version) and reuse.  The cache
        holds the last two contexts (a few MB of fp16 each)."""
        # keyed on the tensor OBJECT (kept alive by the cache, so its storage cannot be recycled under the key) + its version
        # counter (bumped by any in-place write).  Two entries: an unbatched sampler alternates cond / uncond contexts.
        ver = ops.tensor_version(context)
        cache = None
        for cnd in self._kv_caches:
            if cnd["ref"] is context and cnd["ver"] == ver and ver is not None and cnd["rng"] == img_range:
                cache = cnd
                break
        if cache is None:
            cache = {"ref": context, "ver": ver, "rng": img_range}
            self._kv_caches = [cache] + [cnd for cnd in self._kv_caches if cnd["ref"] is not context][:2]
        else:
            self._kv_caches = [cache] + [cnd for cnd in self._kv_caches if cnd is not cache][:2]
        self._kv_cache = cache                     # most recent entry (introspection / tests)

        def project(Q, name, tokens, b):
            k = (id(Q), name, b)
            if k not in cache:
                cache[k] = ops.linear(tokens, Q[name])
            return cache[k]
        return project

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x, timesteps, context=None, features_adapter=None, fs=None, **kwargs):
        """x [B,in_channels,T,H,W], timesteps [B] long, context [B,L,context_dim], fs [B] long -> [B,out_channels,T,H,W]
        in x.dtype (openaimodel3d.py:548-603).  Extra kwargs are accepted and ignored like the reference does."""
        if features_adapter is not None:
            _unsupported("features_adapter")
        if x.is_cuda and context is not None and not torch.cuda.is_current_stream_capturing():
            context = self._canonical_context(context)
            if self._graph_mode:
                return self._forward_graphed(x, timesteps, context, fs, kwargs)
        return self._forward_impl(x, timesteps, context, fs, kwargs)

    def _forward_graphed(self, x, timesteps, context, fs, kwargs):
        ver = ops.tensor_version(context)
        flags = tuple(sorted((k, v if isinstance(v, str) else bool(v)) for k, v in kwargs.items() if k == "cfg_shared_prefix"))
        key = (tuple(x.shape), x.dtype, id(context), ver, fs is None, flags, id(self._comm))
        e = self._graphs.get(key)
        if ver is None or (e is not None and e["ctx"] is not context):
            return self._forward_impl(x, timesteps, context, fs, kwargs)
        if e is None:                                   # first sight: run eagerly (packs weights, fills the K/V cache)
            if len(self._graphs) >= 4:
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = dict(ctx=context, graph=None)
            return self._forward_impl(x, timesteps, context, fs, kwargs)
        dev = x.device
        if e["graph"] is None:                          # second call: capture
            e["x"] = x.clone()
            e["t"] = timesteps.to(device=dev, dtype=torch.int64).clone()
            e["fs"] = None if fs is None else fs.to(device=dev, dtype=torch.int64).clone()
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            n0 = ops.launch_count()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                # the final frame gather is a NCCL collective: keep it out of the capture (the peer-memory exchanges are plain kernels)
                e["out"] = self._forward_impl(e["x"], e["t"], context, e["fs"], kwargs, gather=False)
            e["graph"] = g
            e["launches"] = ops.launch_count() - n0     # kernels of this library inside the graph (launched again by every replay)
            e["kv"] = list(self._kv_caches)             # the captured kernels read these K/V projections: keep them alive
        e["x"].copy_(x)
        e["t"].copy_(timesteps)
        if e["fs"] is not None:
            e["fs"].copy_(fs)
        e["graph"].replay()
        self.graph_replayed_launches += e["launches"]
        out = e["out"]
        if self._comm:
            return self._comm.gather_frames(out, x.shape[2]).to(x.dtype)
        return out.clone()

    def _forward_impl(self, x, timesteps, context, fs, kwargs, gather=True):
        ops.require_cuda(x.device, "viewcrafter_b200.UNetModel")
        P = self._packed or self._pack()
        if P["device"] != x.device:
            raise ops.VcError(f"UNetModel weights are on {P['device']} but the input is on {x.device}")
        comm = self._comm
        T_all = x.shape[2]
        if comm:                                   # frame sharding: this rank owns frames [f0, f1) for every spatial op
            f0, f1 = comm.bind(T_all)
            x_full, x = x, x[:, :, f0:f1]
        B, Cin, T, H, W = x.shape
        dev = x.device
        x32 = x.float().contiguous()
        # cfg_shared_prefix: the caller (DDIMSampler._apply_both, the three-way sampler) asserts that all B (2 or 3) batch rows carry the
        # same x, t, fs and c_concat and differ only in the cross-attention context
        kinds = [Pm["kind"] for Pm in P["input"][1]] if len(P["input"]) > 1 else []
        flag = kwargs.get("cfg_shared_prefix")
        shared = bool(flag) and B in (2, 3) and (comm is None or flag == SHARED_PREFIX_ANY_LAYOUT) and kinds[:2] == ["R", "S"]
        # --- embeddings (fp32) : time_embed(t) + fps_embedding(fs), one row per batch element (frame-invariant) ---
        ts = timesteps.to(device=dev, dtype=torch.int64).contiguous()
        tw = P["time"]
        emb = ops.small_linear(ops.small_linear(ops.timestep_embedding(ts, self.model_channels), tw[0], tw[1]), tw[2], tw[3], silu_in=True)
        if self.fs_condition:
            if fs is None:
                fs = torch.full((B,), self.default_fs, dtype=torch.int64, device=dev)
            fw = P["fps"]
            fs_h = ops.small_linear(ops.timestep_embedding(fs.to(device=dev, dtype=torch.int64).contiguous(), self.model_channels), fw[0], fw[1])
            emb = ops.small_linear(fs_h, fw[2], fw[3], silu_in=True, add=emb)
        # --- context: text[:77] | image tokens; per-frame image tokens when L == 77 + 16*T (openaimodel3d.py:556-560) ---
        ctx16 = ops.cast_f16(context.float().contiguous())
        L = context.shape[1]
        per_frame = (L == 77 + T_all * 16)
        img_lo, img_hi = (77 + 16 * f0, 77 + 16 * f1) if (comm and per_frame) else (77, L)
        ctx = dict(text=[ctx16[b, :77] for b in range(B)], img=[ctx16[b, img_lo:img_hi] for b in range(B)] if L > 77 else None,
                   img_per_frame=per_frame, kv=self._kv_projector(context, (img_lo, img_hi)))
        # --- input latent -> rows [(b t) h w, Cin padded to 8] ---
        cin_pad = max(8, (Cin + 7) // 8 * 8)
        h = torch.zeros((B * T * H * W, cin_pad), device=dev, dtype=torch.float16) if cin_pad != Cin else \
            torch.empty((B * T * H * W, cin_pad), device=dev, dtype=torch.float16)
        ops.ncthw_to_rows(x32, h, 0)

        hs = []
        emb1 = None
        if shared:
            # SURVEY.md App. C.2: all guidance branches see the same x, t, fs and c_concat, so everything before the first
            # cross-attention (input_blocks.0, init_attn, input_blocks.1.0 and input_blocks.1.1 up to attn1) is computed once
            # on one batch element and replicated to B rows; the results are those of the plain B-row forward.  Under frame
            # sharding the prefix's layout switches run at B=1.
            emb1 = emb[:1].contiguous()
            h = h[:T * H * W]
            h, H, W = self._run_stage(P["input"][0], h, None, emb1, ctx, 1, T, H, W)
            if self.addition_attention:
                h, H, W = self._run_stage(P["init_attn"], h, None, emb1, ctx, 1, T, H, W)
            hs.append(torch.cat([h] * B, 0))       # a copy: also detaches the skip from a reusable peer receive buffer
        for i, stage in enumerate(P["input"]):
            if i == 0 and shared:
                continue
            h, H, W = self._run_stage(stage, h, None, emb, ctx, B, T, H, W, emb1=emb1 if i == 1 else None)
            if i == 0 and self.addition_attention:
                h, H, W = self._run_stage(P["init_attn"], h, None, emb, ctx, B, T, H, W)
            if comm and getattr(comm, "owns", None) and comm.owns(h):
                h = h.clone()                      # a skip outlives the reusable peer receive buffer it was delivered in
            hs.append(h)
        h, H, W = self._run_stage(P["middle"], h, None, emb, ctx, B, T, H, W)
        for stage in P["output"]:
            h, H, W = self._run_stage(stage, h, hs.pop(), emb, ctx, B, T, H, W)
        y = ops.conv3x3(ops.groupnorm(h, B * T, *P["out_gn"], 1e-5, True), B * T, H, W, P["out_w"], bias=P["out_b"], out_f32=True)
        out = ops.rows_to_ncthw(y, B, self.out_channels, T, H, W)
        if comm:                                   # every rank needs the whole prediction for the (global-std) DDIM update
            if not gather:
                return out                            # this rank's frames only (the graph path gathers after the replay)
            out = comm.gather_frames(out, T_all)
        return out.to(x.dtype)
