"""VideoUNet: drop-in for `sgm.modules.diffusionmodules.video_model.VideoUNet` (video_model.py:84-501).

Same constructor kwargs, same `state_dict` keys/shapes, same `forward` signature and output -- but the
module is a parameter container plus a *compiled launch plan*: for a given (batch, H, W, T) the whole forward
is a flat list of C-ABI kernel launches (hi3d_gemm / hi3d_groupnorm_silu / hi3d_layernorm /
hi3d_attention_d64 / hi3d_temporal_attention_d64 ...) over pre-allocated channels-last fp16 buffers with
pre-baked parameter blocks, replayable under a CUDA graph.  There is no per-op nn.Module graph and no
PyTorch compute on the path.

Algebraic folds relative to the reference graph (all exact in real arithmetic; SURVEY.md F7, App. E):
  * single-token cross-attention attn2(x, ctx) == to_out(to_v(ctx)) -> a per-sample bias row added in the
    epilogue of the attn1 output projection (to_q / to_k / norm2 are dead compute);
  * time_pos_embed(arange(T)) depends only on T -> computed once per plan;
  * label_emb(y) and the cross-attention rows are step-invariant -> `prepare_conditioning` runs them once
    per video; the generic `forward()` recomputes them every call (it cannot know the caller's loop);
  * 1x1 skip convs are extra K-segments of the second 3x3 conv GEMM; th.cat([h, hs.pop()]) is never
    materialised (two K-segments per tap); AlphaBlender and every residual add live in GEMM epilogues;
  * "(b t) s c <-> (b s) t c" rearranges of the temporal transformer are pure addressing.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import ops, pack
from .spec import Layer, UNetConfig, unet_param_shapes, unet_plan

F16 = torch.float16
CIN_PAD = 64     # UNet input channels are zero-padded to one 64-wide K segment per tap
COUT_PAD = 8     # final conv output channels padded to the engine's N granularity


class _ParamTree(nn.Module):
    """Nested holder so parameters get the reference's dotted names (input_blocks.1.0.in_layers.2.weight ...)."""

    def put(self, dotted: str, p: nn.Parameter):
        parts = dotted.split(".")
        node = self
        for q in parts[:-1]:
            if q not in node._modules:
                node.add_module(q, _ParamTree())
            node = node._modules[q]
        node.register_parameter(parts[-1], p)


class Arena:
    """Named scratch buffers: one allocation per tag, sized to the largest request, handed out as views.
    Tags listed in `symm_tags` are allocated as symmetric peer memory (peer.SymmBuffer): every rank of a frame-sharded
    run holds the same buffer at the same tag and can address the other ranks' copies (`peers(tag)`)."""

    def __init__(self, device, peer_group=None, symm_tags=()):
        self.device = device
        self.req: Dict[str, int] = {}
        self.bufs: Dict[str, torch.Tensor] = {}
        self.views: List[Tuple[str, int, int, list]] = []
        self.peer_group, self.symm_tags = peer_group, tuple(symm_tags)
        self.symm: Dict[str, object] = {}

    def want(self, tag: str, rows: int, cols: int) -> "LazyBuf":
        n = rows * cols
        self.req[tag] = max(self.req.get(tag, 0), n)
        return LazyBuf(self, tag, rows, cols)

    def materialise(self):
        for tag, n in sorted(self.req.items()):           # sorted: every rank allocates the symmetric tags in the same order
            if tag not in self.bufs or self.bufs[tag].numel() < n:
                if self.peer_group is not None and tag in self.symm_tags:
                    sb = self.peer_group.alloc(n * 2)
                    self.symm[tag] = sb
                    self.bufs[tag] = sb.view(F16)[:n]
                else:
                    self.bufs[tag] = torch.zeros(n, dtype=F16, device=self.device)

    def peers(self, tag: str):
        """peer.SymmBuffer of a symmetric tag (views of a tag start at offset 0, so the peers' base pointers address the same
        rows on every rank)."""
        return self.symm[tag]

    def get(self, tag: str, rows: int, cols: int) -> torch.Tensor:
        return self.bufs[tag][: rows * cols].view(rows, cols)

    def nbytes(self) -> int:
        return sum(b.numel() * 2 for b in self.bufs.values())


class LazyBuf:
    __slots__ = ("arena", "tag", "rows", "cols")

    def __init__(self, arena, tag, rows, cols):
        self.arena, self.tag, self.rows, self.cols = arena, tag, rows, cols

    @property
    def t(self) -> torch.Tensor:
        return self.arena.get(self.tag, self.rows, self.cols)


class StatsBuf:
    """One GroupNorm statistics table fp32 [n_img, units, 2] inside the plan's statistics arena (zeroed once per forward)."""
    __slots__ = ("plan", "off", "n_img", "units")

    def __init__(self, plan, off, n_img, units):
        self.plan, self.off, self.n_img, self.units = plan, off, n_img, units

    @property
    def t(self) -> torch.Tensor:
        return self.plan.stats_arena[self.off:self.off + self.n_img * self.units * 2]


class VideoUNet(nn.Module):
    def __init__(self, **kwargs):
        super().__init__()
        self.cfg = UNetConfig.from_kwargs(**kwargs)
        self.plan_desc = unet_plan(self.cfg)
        self.in_channels, self.out_channels = self.cfg.in_channels, self.cfg.out_channels
        self.model_channels, self.num_classes = self.cfg.model_channels, self.cfg.num_classes
        tree = _ParamTree()
        for name, shp in unet_param_shapes(self.cfg).items():
            tree.put(name, nn.Parameter(torch.empty(shp), requires_grad=False))
        # expose the reference's top-level attribute names (time_embed, label_emb, input_blocks, ...)
        for k, m in tree._modules.items():
            self.add_module(k, m)
        self._packed: Optional[dict] = None
        self._plans: Dict[tuple, "_Plan"] = {}
        self.engine = os.environ.get("HI3D_ENGINE", "tc5")     # "tc5" = tcgen05/TMEM/TMA engine, "mma" = mma.sync engine
        # packed weights, launch plans and captured graphs derive from the parameters: ANY load that reaches this module
        # -- its own load_state_dict or a parent's (DiffusionEngine.init_from_ckpt recurses through
        # _load_from_state_dict and never calls the override below) -- must drop them
        self._register_load_state_dict_pre_hook(lambda *a, **k: self._invalidate())

    # ---- parameter lifecycle ---------------------------------------------------------------------------
    def _invalidate(self):
        self._packed = None
        self._plans = {}

    def _apply(self, fn, *a, **k):
        self._invalidate()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._invalidate()
        return super().load_state_dict(*a, **k)

    def set_engine(self, engine: str):
        if engine not in ("mma", "tc5"):
            raise ValueError(engine)
        if engine != self.engine:
            self.engine = engine
            self._plans = {}

    @property
    def device(self):
        return self.out._modules["0"].weight.device

    # ---- weight packing ----------------------------------------------------------------------------------
    def _pack(self) -> dict:
        if self._packed is not None:
            return self._packed
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("hi3d_official_b200.VideoUNet computes only on CUDA (B200); call .cuda() first -- "
                               "there is no CPU fallback")
        P: dict = {}
        lin, bias = pack.pack_linear, pack.pack_bias

        def f32(k):
            return sd[k].float().contiguous()

        def pb(k):
            return sd[k].float().contiguous()
        mc = self.cfg.model_channels
        P["time_embed.0"] = (lin(sd["time_embed.0.weight"]), pb("time_embed.0.bias"))
        P["time_embed.2"] = (lin(sd["time_embed.2.weight"]), pb("time_embed.2.bias"))
        P["label_emb.0"] = (lin(sd["label_emb.0.0.weight"]), pb("label_emb.0.0.bias"))
        P["label_emb.2"] = (lin(sd["label_emb.0.2.weight"]), pb("label_emb.0.2.bias"))
        emb_w, emb_b, emb_off, off = [], [], {}, 0
        layers = [L for blk in self.plan_desc.input_blocks + [self.plan_desc.middle] + self.plan_desc.output_blocks
                  for L in blk]
        for L in layers:
            n = L.name
            if L.kind == "conv_in":
                P[n] = (pack.pack_conv2d(sd[n + "weight"], cin_pad=CIN_PAD), pb(n + "bias"))
            elif L.kind == "down":
                P[n] = (pack.pack_conv2d(sd[n + "op.weight"]), pb(n + "op.bias"))
            elif L.kind == "up":
                P[n] = (pack.pack_upconv_parity(sd[n + "conv.weight"]), pb(n + "conv.bias"))
            elif L.kind == "res":
                for sub, tconv in (("", False), ("time_stack.", True)):
                    q = n + sub
                    pk = pack.pack_conv3d_t if tconv else pack.pack_conv2d
                    P[q + "gn1"] = (f32(q + "in_layers.0.weight"), f32(q + "in_layers.0.bias"))
                    P[q + "conv1"] = (pk(sd[q + "in_layers.2.weight"]), pb(q + "in_layers.2.bias"))
                    P[q + "gn2"] = (f32(q + "out_layers.0.weight"), f32(q + "out_layers.0.bias"))
                    w2, b2 = pk(sd[q + "out_layers.3.weight"]), pb(q + "out_layers.3.bias")
                    if q + "skip_connection.weight" in sd:
                        w2 = pack.cat_k(w2, pack.pack_conv2d(sd[q + "skip_connection.weight"]))
                        b2 = b2 + pb(q + "skip_connection.bias")
                    P[q + "conv2"] = (w2, b2.contiguous())
                    emb_w.append(lin(sd[q + "emb_layers.1.weight"]))
                    emb_b.append(pb(q + "emb_layers.1.bias"))
                    emb_off[q] = (off, emb_w[-1].shape[0])
                    off += emb_w[-1].shape[0]
                P[n + "alpha"] = float(torch.sigmoid(sd[n + "time_mixer.mix_factor"].float()).item())
            elif L.kind == "attn":
                P[n + "norm"] = (f32(n + "norm.weight"), f32(n + "norm.bias"))
                P[n + "proj_in"] = (lin(sd[n + "proj_in.weight"]), pb(n + "proj_in.bias"))
                P[n + "proj_out"] = (lin(sd[n + "proj_out.weight"]), pb(n + "proj_out.bias"))
                P[n + "tpe0"] = (lin(sd[n + "time_pos_embed.0.weight"]), pb(n + "time_pos_embed.0.bias"))
                P[n + "tpe2"] = (lin(sd[n + "time_pos_embed.2.weight"]), pb(n + "time_pos_embed.2.bias"))
                P[n + "alpha"] = float(torch.sigmoid(sd[n + "time_mixer.mix_factor"].float()).item())
                for d in range(self.cfg.transformer_depth):
                    for q, temporal in ((n + f"transformer_blocks.{d}.", False), (n + f"time_stack.{d}.", True)):
                        for nm in ("norm1", "norm3") + (("norm_in",) if temporal else ()):
                            P[q + nm] = (f32(q + nm + ".weight"), f32(q + nm + ".bias"))
                        P[q + "qkv"] = torch.cat([lin(sd[q + "attn1.to_q.weight"]), lin(sd[q + "attn1.to_k.weight"]),
                                                  lin(sd[q + "attn1.to_v.weight"])], 0).contiguous()
                        P[q + "to_out"] = (lin(sd[q + "attn1.to_out.0.weight"]), pb(q + "attn1.to_out.0.bias"))
                        P[q + "ca_v"] = lin(sd[q + "attn2.to_v.weight"])
                        P[q + "ca_out"] = (lin(sd[q + "attn2.to_out.0.weight"]), pb(q + "attn2.to_out.0.bias"))
                        for ff in ("ff",) + (("ff_in",) if temporal else ()):
                            P[q + ff + "1"] = pack.pack_geglu(sd[q + ff + ".net.0.proj.weight"],
                                                              sd[q + ff + ".net.0.proj.bias"])
                            P[q + ff + "2"] = (lin(sd[q + ff + ".net.2.weight"]), pb(q + ff + ".net.2.bias"))
        P["emb_all"] = (torch.cat(emb_w, 0).contiguous(), torch.cat(emb_b, 0).contiguous())
        P["emb_off"], P["emb_total"] = emb_off, off
        P["out.gn"] = (f32("out.0.weight"), f32("out.0.bias"))
        P["out.conv"] = (pack.pack_conv2d(sd["out.2.weight"], cout_pad=COUT_PAD),
                         pack.pack_bias(sd["out.2.bias"], self.cfg.out_channels, COUT_PAD))
        self._packed = P
        return P

    # ---- plans --------------------------------------------------------------------------------------------
    def plan_key(self, N: int, H: int, W: int, T: int, shard: Optional[Tuple[int, int]] = None) -> tuple:
        """Key of the launch plan get_plan returns now: the shape, the engine and the deterministic-mode switch
        (ops.deterministic(), read here), so that toggling the switch builds a fresh plan instead of replaying a stale one."""
        key = (N, H, W, T, self.engine, ops.deterministic())
        return key if shard is None else key + (tuple(shard),)

    def get_plan(self, N: int, H: int, W: int, T: int, shard: Optional[Tuple[int, int]] = None) -> "_Plan":
        """shard = (rank, world): frame-sharded plan -- N = B * T local samples, this rank owns frames
        [rank*T, (rank+1)*T) of clips of world*T frames (SURVEY 8e; needs an initialised torch.distributed group)."""
        key = self.plan_key(N, H, W, T, shard)
        if key not in self._plans:
            self._plans[key] = _Plan(self, N, H, W, T, shard=shard, det=key[5])
        return self._plans[key]

    # ---- reference-compatible forward ------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x: torch.Tensor, timesteps: torch.Tensor, context: Optional[torch.Tensor] = None,
                y: Optional[torch.Tensor] = None, time_context: Optional[torch.Tensor] = None,
                num_video_frames: Optional[int] = None, image_only_indicator: Optional[torch.Tensor] = None):
        assert (y is not None) == (self.num_classes is not None), \
            "must specify y if and only if the model is class-conditional"
        assert context is not None and num_video_frames is not None
        if time_context is not None:
            raise NotImplementedError("explicit time_context: Hi3D configs use use_spatial_context=True")
        if image_only_indicator is not None and bool(image_only_indicator.any()):
            raise NotImplementedError("image_only_indicator != 0 (image-only frames) is outside the Hi3D hot path")
        N, Cin, H, W = x.shape
        assert Cin == self.in_channels, f"expected {self.in_channels} input channels, got {Cin}"
        plan = self.get_plan(N, H, W, num_video_frames)
        plan.prepare_conditioning(context, y)
        ops.nchw_to_nhwc(x.contiguous(), plan.xin.t.view(N, H, W, CIN_PAD))
        plan.set_timesteps(timesteps)
        plan.run()
        out = torch.empty(N, self.out_channels, H, W, dtype=F16, device=x.device)
        ops.nhwc_to_nchw(plan.net_out.t, out)
        return out


# ==================================================================================================================
class _Plan:
    """Flat launch list for one (N, H, W, T): buffers, pre-baked GEMM parameter blocks, per-step entry points."""

    def __init__(self, net: VideoUNet, N: int, H: int, W: int, T: int, shard: Optional[Tuple[int, int]] = None,
                 det: bool = False):
        self.det = det                 # deterministic GroupNorm statistics (ops.deterministic())
        self.shard = None if shard is None or shard[1] == 1 else (int(shard[0]), int(shard[1]))
        self.rank, self.world = self.shard if self.shard else (0, 1)
        self.Tg = T * self.world                     # frames per clip over all ranks
        if N % T:
            raise ValueError(f"batch {N} is not a multiple of num_video_frames {T}")
        if T * (1 if shard is None else int(shard[1])) > 16:
            raise NotImplementedError("temporal attention kernel supports T <= 16 frames")
        nlev = len(net.cfg.channel_mult)
        if H % (1 << (nlev - 1)) or W % (1 << (nlev - 1)):
            raise ValueError(f"H, W = {H}, {W} must be divisible by {1 << (nlev - 1)}")
        self.net, self.N, self.H, self.W, self.T, self.B = net, N, H, W, T, N // T
        self.P = net._pack()
        self.dev = net.device
        self.engine = net.engine
        self.attn_engine = os.environ.get("HI3D_ATTN_ENGINE", net.engine)
        # frame sharding: how the three cross-frame ops exchange data (SURVEY 8e).  "peer" (default) = peer-memory loads /
        # stores inside the consuming / producing kernels + one flag-barrier kernel per exchange point, CUDA-graph
        # capturable; "nccl" = torch.distributed collectives (dist.py), eager.
        self.exchange_mode = os.environ.get("HI3D_SHARD_EXCHANGE", "peer") if self.shard else None
        if self.exchange_mode not in (None, "peer", "nccl"):
            raise ValueError(f"HI3D_SHARD_EXCHANGE={self.exchange_mode!r}: expected 'peer' or 'nccl'")
        self.peer = None
        if self.exchange_mode == "peer":
            from . import peer as _peer
            forced = "HI3D_SHARD_EXCHANGE" in os.environ
            try:
                self.peer = _peer.get_group(self.rank, self.world, self.dev)
                ok = 1
            except Exception as e:          # no peer-to-peer access between the GPUs of this box (IPC open fails on every rank)
                if forced:
                    raise
                ok, why = 0, e
            if not forced:
                # the ranks must agree: one rank on NCCL and another on peer memory would deadlock
                import torch.distributed as _dist
                flag = torch.tensor([ok], dtype=torch.int32, device=self.dev)
                _dist.all_reduce(flag, op=_dist.ReduceOp.MIN)
                if int(flag.item()) == 0:
                    if self.rank == 0:
                        import sys
                        print("hi3d: peer-memory exchange unavailable on this box"
                              + (f" ({why})" if not ok else " (on another rank)") + "; frame sharding falls back to NCCL exchanges",
                              file=sys.stderr)
                    self.peer, self.exchange_mode = None, "nccl"
        self.arena = Arena(self.dev, self.peer, ("qkv", "att", "ghalo") if self.peer is not None else ())
        # GroupNorm statistics from the producing GEMM epilogues (hi3d_gemm_params::gn_stats): every GroupNorm is ONE launch
        # (apply); HI3D_GN_FUSED=0 keeps the separate statistics pass (stats + finalize + apply)
        self.gn_unit = net.cfg.model_channels // 32
        self.gn_fused = (os.environ.get("HI3D_GN_FUSED", "1") != "0" and net.cfg.model_channels % 32 == 0
                         and net.cfg.model_channels * max(net.cfg.channel_mult) // self.gn_unit <= 256)
        self._stats_floats = 0
        self.stats_arena = None
        # deterministic mode: scratch for the statistics partials, shared by every producer (a table is dead once folded)
        self._part_floats = 0
        self.gn_part = None
        self._nvtx_open = False
        self.steps: List = []          # main per-step launch list (built lazily as (kind, builder) then baked)
        self._build: List = []         # deferred builders, run after the arena is materialised
        self._cond_build: List = []
        self.cond_steps: List = []
        self.flops = 0.0
        self._graph = None
        cfg = net.cfg
        mc, E = cfg.model_channels, cfg.model_channels * 4
        dev = self.dev
        # small persistent (non-arena) tensors
        self.t_in = torch.zeros(N, dtype=torch.float32, device=dev)
        self.temb = torch.zeros(N, mc, dtype=F16, device=dev)
        self.e1 = torch.zeros(N, E, dtype=F16, device=dev)
        self.emb_act = torch.zeros(N, E, dtype=F16, device=dev)
        self.emb_all = torch.zeros(N, self.P["emb_total"], dtype=F16, device=dev)
        self.label = torch.zeros(N, E, dtype=F16, device=dev)
        self.y_in = torch.zeros(N, cfg.adm_in_channels, dtype=F16, device=dev)
        self.y_h = torch.zeros(N, E, dtype=F16, device=dev)
        self.ctx_in = torch.zeros(N, cfg.context_dim, dtype=F16, device=dev)
        self.ctx_first = torch.zeros(self.B, cfg.context_dim, dtype=F16, device=dev)
        self.gn_ws = ops.groupnorm_ws(N, dev)
        self.frame_idx = torch.arange(T, dtype=torch.float32, device=dev) + float(self.rank * T)   # global frame ids
        self.gn_sums = torch.zeros(self.B, 32, 2, dtype=torch.float32, device=dev)               # sharded temporal GN
        self.gn_sums_local = torch.zeros(self.B, 32, 2, dtype=torch.float32, device=dev)
        self._cond_key = None
        self._compile()
        if self.peer is not None:
            # ranks build their plans (weight packing, tensor maps) at different speeds: meet on the host once, so that the
            # first exchange kernel of the step does not spin for seconds on a rank that is still compiling
            import torch.distributed as dist
            torch.cuda.synchronize()
            dist.barrier(group=self.peer.pg)

    # ---- helpers -----------------------------------------------------------------------------------------------
    # Statistics in the epilogue are free where the main loop hides the epilogue (3x3 convs, wide temporal convs, K >= 1920 --
    # the same threshold as the CTA-pair rule) and cost MORE than a separate statistics pass on the epilogue-bound short-K
    # GEMMs (measured, profiles/r02_gn_epilogue_notes.txt: temporal conv C=320 +165 us per launch against 87 us for the
    # pass): those keep the pass (hi3d_groupnorm_unit_stats, same table), still one launch less than r01's stats + finalize.
    GN_FUSE_MIN_K = 1920

    def _gemm(self, lst, segs_fn, W, out: LazyBuf, M, gn_defer: bool = False, **kw):
        """Defer Gemm construction until buffers exist. segs_fn() -> list[SegSpec]; tensor kwargs may be LazyBuf.
        gn_defer: the caller adds the separate statistics pass itself (several launches fill one tensor)."""
        post = None
        if kw.get("gn_stats") is not None:
            self._need_partials(kw["gn_stats"], out)
        if kw.get("gn_stats") is not None and W.shape[1] < self.GN_FUSE_MIN_K:
            st, unit, rows = kw.pop("gn_stats"), kw.pop("gn_unit"), kw.pop("gn_rows")
            if not gn_defer:
                post = lambda: (lambda: ops.groupnorm_unit_stats(out.t, st.n_img, (out.rows // st.n_img), unit, st.t, self.gn_part))

        def build():
            k2 = {}
            for k, v in kw.items():
                k2[k] = v.t if isinstance(v, (LazyBuf, StatsBuf)) else v
            if self.det and "gn_stats" in k2:
                k2["gn_partials"] = self.gn_part
            g = ops.Gemm(segs_fn(), W, out.t if isinstance(out, LazyBuf) else out, M, engine=self.engine, **k2)
            self.flops += g.flops if lst is self._build else 0.0
            return g
        lst.append(build)
        if post is not None:
            fn = post()
            fn.kind, fn.bytes = "groupnorm", 2.0 * out.rows * out.cols
            lst.append(lambda fn=fn: fn)

    def _mark(self, name: str):
        """HI3D_NVTX=1: an NVTX range per layer of the launch plan (block name as in the state dict), so that ncu / nsys
        captures can be filtered and read by layer (`ncu --nvtx --nvtx-include "input_blocks.1.1.*/"`).  Host-side marker
        calls only; not part of CUDA-graph replays (profile with HI3D_CUDA_GRAPH=0)."""
        if os.environ.get("HI3D_NVTX", "0") == "1":
            def m(name=name):
                torch.cuda.nvtx.range_pop() if self._nvtx_open else None
                torch.cuda.nvtx.range_push(name)
                self._nvtx_open = True
            self._call(self._build, m, kind="marker")

    def _need_partials(self, st: StatsBuf, out: LazyBuf):
        """Deterministic mode: grow the partials scratch to what the producer of `st` (over the tensor `out`) needs."""
        if self.det:
            self._part_floats = max(self._part_floats, ops.groupnorm_partials_floats(st.n_img, out.rows // st.n_img, out.cols,
                                                                                     self.gn_unit))

    def _stats(self, n_img: int, C: int) -> Optional[StatsBuf]:
        if not self.gn_fused:
            return None
        sb = StatsBuf(self, self._stats_floats, n_img, C // self.gn_unit)
        self._stats_floats += n_img * (C // self.gn_unit) * 2
        return sb

    def _gnkw(self, stats: Optional[StatsBuf], rows_per_img: int) -> dict:
        """Gemm kwargs that make its epilogue accumulate the GroupNorm statistics of its output into `stats`."""
        return {} if stats is None else dict(gn_stats=stats, gn_unit=self.gn_unit, gn_rows=rows_per_img)

    def _gn(self, lst, srcs, n_samples: int, rows_per_sample: int, ips: int, gb, eps: float, silu: bool, y: LazyBuf,
            count_rows: Optional[int] = None, **halo):
        """GroupNorm(32)[+SiLU] of the channel concat of srcs = [(LazyBuf, C, StatsBuf | None), ...] into y.
        Fused statistics: one apply launch reading the producers' unit tables; otherwise stats + finalize + apply."""
        gam, bet = gb
        x1, c1, st1 = srcs[0]
        x2, c2, st2 = srcs[1] if len(srcs) > 1 else (None, 0, None)
        C = c1 + c2
        M = n_samples * rows_per_sample
        ws = self.gn_ws
        if self.gn_fused and st1 is not None and (x2 is None or st2 is not None):
            self._call(lst, lambda: ops.groupnorm_apply_stats(
                x1.t, st1.t, x2.t if x2 else None, st2.t if x2 else None, self.gn_unit, n_samples, rows_per_sample, ips,
                count_rows or rows_per_sample, gam, bet, eps, silu, y.t, **halo), kind="groupnorm", bytes=4.0 * M * C)
        else:
            assert not halo and count_rows is None
            self._call(lst, lambda: ops.groupnorm_silu(x1.t, x2.t if x2 else None, n_samples, rows_per_sample, gam, bet, eps,
                                                       silu, y.t, ws, self.det), kind="groupnorm", bytes=6.0 * M * C)

    def _call(self, lst, fn, **meta):
        """meta: kind / flops / bytes = algorithmic work of the launch (read by bench.py's breakdown)."""
        for k, v in meta.items():
            setattr(fn, k, v)
        lst.append(lambda: fn)

    def _compile(self):
        net, P, cfg = self.net, self.P, self.net.cfg
        N, T, B = self.N, self.T, self.B
        A = self.arena
        H, W = self.H, self.W
        mc, E = cfg.model_channels, cfg.model_channels * 4
        bl = self._build

        # ---------------- per-step embedding path (video_model.py:456-469, openaimodel.py:341) ----------------
        self._call(bl, lambda: ops.timestep_embedding(self.t_in, mc, self.temb))
        self._gemm(bl, lambda: [ops.SegSpec(self.temb)], P["time_embed.0"][0], self.e1, N, bias=P["time_embed.0"][1],
                   act=ops.ACT_SILU)
        self._gemm(bl, lambda: [ops.SegSpec(self.e1)], P["time_embed.2"][0], self.emb_act, N,
                   bias=P["time_embed.2"][1], rowbias=self.label, rb_div=1, rb_mod=N, act=ops.ACT_SILU)
        self._gemm(bl, lambda: [ops.SegSpec(self.emb_act)], P["emb_all"][0], self.emb_all, N, bias=P["emb_all"][1])

        # ---------------- conditioning path (once per video) ----------------
        cl = self._cond_build
        self._gemm(cl, lambda: [ops.SegSpec(self.y_in)], P["label_emb.0"][0], self.y_h, N, bias=P["label_emb.0"][1],
                   act=ops.ACT_SILU)
        self._gemm(cl, lambda: [ops.SegSpec(self.y_h)], P["label_emb.2"][0], self.label, N, bias=P["label_emb.2"][1])

        # ---------------- main body ----------------
        if self.gn_fused:      # first launch of every forward: the statistics tables the epilogues accumulate into
            self._call(bl, lambda: self.stats_arena.zero_(), kind="memset")
        self.xin = A.want("xin", N * H * W, CIN_PAD)
        hs: List[tuple] = []          # (buffer, C, h, w, stats)
        cur: tuple = None
        self._pp = 0

        def next_out(rows, C, persist_tag=None):
            if persist_tag:
                return A.want(persist_tag, rows, C)
            self._pp ^= 1
            return A.want(f"blk{self._pp}", rows, C)

        h, w = H, W
        for bi, blk in enumerate(self.plan_desc_blocks("input")):
            for li, L in enumerate(blk):
                last = li == len(blk) - 1
                tag = f"hs{bi}" if last else None
                if L.kind == "conv_in":
                    out, st = next_out(N * h * w, L.cout, tag), self._stats(N, L.cout)
                    self._conv(bl, [self.xin], P[L.name], out, h, w, h, w, **self._gnkw(st, h * w))
                elif L.kind == "res":
                    out, st = next_out(N * h * w, L.cout, tag), self._stats(N, L.cout)
                    self._resblock(L, [cur], out, st, h, w)
                elif L.kind == "attn":
                    out, st = next_out(N * h * w, L.cout, tag), self._stats(N, L.cout)
                    self._transformer(L, cur, out, st, h, w)
                elif L.kind == "down":
                    out, st = next_out(N * (h // 2) * (w // 2), L.cout, tag), self._stats(N, L.cout)
                    self._conv(bl, [cur[0]], P[L.name], out, h // 2, w // 2, h, w, stride=2, **self._gnkw(st, (h // 2) * (w // 2)))
                    h, w = h // 2, w // 2
                cur = (out, L.cout, h, w, st)
            hs.append(cur)
        for L in self.net.plan_desc.middle:
            out, st = next_out(N * h * w, L.cout), self._stats(N, L.cout)
            if L.kind == "res":
                self._resblock(L, [cur], out, st, h, w)
            else:
                self._transformer(L, cur, out, st, h, w)
            cur = (out, L.cout, h, w, st)
        for blk in self.plan_desc_blocks("output"):
            skip = hs.pop()
            assert (skip[2], skip[3]) == (h, w)
            srcs = [cur, skip]
            for L in blk:
                if L.kind == "res":
                    out, st = next_out(N * h * w, L.cout), self._stats(N, L.cout)
                    self._resblock(L, srcs, out, st, h, w)
                elif L.kind == "attn":
                    out, st = next_out(N * h * w, L.cout), self._stats(N, L.cout)
                    self._transformer(L, cur, out, st, h, w)
                elif L.kind == "up":
                    out, st = next_out(N * 4 * h * w, L.cout), self._stats(N, L.cout)
                    self._upconv(bl, cur[0], P[L.name], out, h, w, **self._gnkw(st, h * w))
                    h, w = 2 * h, 2 * w
                cur = (out, L.cout, h, w, st)
        # out: GN32 -> SiLU -> conv3x3 (video_model.py:436-440,500-501)
        M = N * h * w
        g = A.want("gn", M, cur[1])
        self._gn(bl, [(cur[0], cur[1], cur[4])], N, h * w, 1, P["out.gn"], 1e-5, True, g)
        self.net_out = A.want("net_out", M, COUT_PAD)
        self._conv(bl, [g], P["out.conv"], self.net_out, h, w, h, w)

        # ---------------- materialise buffers, bake launches ----------------
        A.materialise()
        if self.gn_fused:
            self.stats_arena = torch.zeros(max(self._stats_floats, 2), dtype=torch.float32, device=self.dev)
        if self.det:
            self.gn_part = torch.empty(max(self._part_floats, 4), dtype=torch.float32, device=self.dev)
        self.steps = [b() for b in self._build]
        self.cond_steps = [b() for b in self._cond_build]
        self._build = self._cond_build = None

    def plan_desc_blocks(self, which):
        return self.net.plan_desc.input_blocks if which == "input" else self.net.plan_desc.output_blocks

    # ---- layer emitters ----------------------------------------------------------------------------------------
    def _conv(self, lst, srcs: List[LazyBuf], wb, out: LazyBuf, ho, wo, hs_, ws_, stride=1, ups=0, **kw):
        Wt, b = wb
        M = self.N * ho * wo
        self._gemm(lst, lambda: ops.conv_taps([s.t for s in srcs]), Wt, out, M, mode=ops.ROWS_CONV2D,
                   geom=dict(Ho=ho, Wo=wo, Hs=hs_, Ws=ws_, stride=stride, ups=ups), bias=b, **kw)

    def _upconv(self, lst, src: LazyBuf, wb, out: LazyBuf, h, w, n_img=None, **kw):
        """Upsample (nearest x2) + conv3x3 (openaimodel.py:154-156) as four parity-class 2x2 convs on the source
        grid with pre-summed taps (pack.pack_upconv_parity): no upsampled tensor, 4/9 of the FLOPs."""
        parity, b = wb
        n_img = self.N if n_img is None else n_img
        M = n_img * h * w
        fused = True
        for (py, px), (Wt, shifts) in parity.items():
            fused = Wt.shape[1] >= self.GN_FUSE_MIN_K
            self._gemm(lst, lambda shifts=shifts: [ops.SegSpec(src.t, dy=sy, dx=sx) for sy, sx in shifts], Wt, out, M,
                       mode=ops.ROWS_CONV2D, geom=dict(Ho=h, Wo=w, Hs=h, Ws=w, out_up=1, out_py=py, out_px=px), bias=b,
                       gn_defer=True, **kw)
        if kw.get("gn_stats") is not None and not fused:       # one statistics pass over the tensor the four launches filled
            st, unit = kw["gn_stats"], kw["gn_unit"]
            self._call(lst, lambda: ops.groupnorm_unit_stats(out.t, st.n_img, out.rows // st.n_img, unit, st.t, self.gn_part),
                       kind="groupnorm", bytes=2.0 * out.rows * out.cols)

    def _emb_slice(self, q):
        off, n = self.P["emb_off"][q]
        return self.emb_all[:, off:off + n]

    def _resblock(self, L: Layer, srcs: List[tuple], out: LazyBuf, out_stats, h: int, w: int):
        self._mark(L.name + "VideoResBlock")
        return self._resblock_impl(L, srcs, out, out_stats, h, w)

    def _resblock_impl(self, L: Layer, srcs: List[tuple], out: LazyBuf, out_stats, h: int, w: int):
        """VideoResBlock (video_model.py:62-81) = spatial ResBlock (openaimodel.py:328-354) + temporal ResBlock
        (dims=3, kernel (3,1,1), GroupNorm over (C/32, T, H, W)) + AlphaBlender, as 4 GN launches + 4 GEMMs.
        srcs = [(buffer, C, h, w, stats), ...] (two entries = the skip concat); every GEMM whose output feeds a GroupNorm
        accumulates that GroupNorm's statistics in its epilogue (`out_stats` for the block output)."""
        P, A, bl, N, T, B = self.P, self.arena, self._build, self.N, self.T, self.B
        n = L.name
        HW = h * w
        M = N * HW
        cs = [s_[1] for s_ in srcs]
        cin, cout = sum(cs), L.cout
        x1 = srcs[0][0]
        x2 = srcs[1][0] if len(srcs) > 1 else None
        g_in = A.want("gn", M, cin)
        hbuf = A.want("h", M, cout)
        g_mid = A.want("gn", M, cout)
        xs = A.want("xs", M, cout)
        st_h1, st_xs, st_h2 = self._stats(N, cout), self._stats(N, cout), self._stats(N, cout)
        # -- spatial half
        self._gn(bl, [(s_[0], s_[1], s_[4]) for s_ in srcs], N, HW, 1, P[n + "gn1"], 1e-5, True, g_in)
        emb1 = self._emb_slice(n)
        self._gemm(bl, lambda: ops.conv_taps([g_in.t]), P[n + "conv1"][0], hbuf, M, mode=ops.ROWS_CONV2D,
                   geom=dict(Ho=h, Wo=w, Hs=h, Ws=w), bias=P[n + "conv1"][1], rowbias=emb1, rb_div=HW, rb_mod=N,
                   **self._gnkw(st_h1, HW))
        self._gn(bl, [(hbuf, cout, st_h1)], N, HW, 1, P[n + "gn2"], 1e-5, True, g_mid)
        if cin != cout:
            self._gemm(bl, lambda: ops.conv_taps([g_mid.t]) + [ops.SegSpec(s_[0].t) for s_ in srcs], P[n + "conv2"][0], xs, M,
                       mode=ops.ROWS_CONV2D, geom=dict(Ho=h, Wo=w, Hs=h, Ws=w), bias=P[n + "conv2"][1], **self._gnkw(st_xs, HW))
        else:
            assert x2 is None
            self._gemm(bl, lambda: ops.conv_taps([g_mid.t]), P[n + "conv2"][0], xs, M, mode=ops.ROWS_CONV2D,
                       geom=dict(Ho=h, Wo=w, Hs=h, Ws=w), bias=P[n + "conv2"][1], residual=x1, **self._gnkw(st_xs, HW))
        # -- temporal half: statistics over (T, H, W) per clip, 3-tap conv along frames
        q = n + "time_stack."
        g3, b3 = P[q + "gn1"]
        g4, b4 = P[q + "gn2"]
        emb2 = self._emb_slice(q)
        ws = self.gn_ws
        if self.shard is None:
            self._gn(bl, [(xs, cout, st_xs)], B, T * HW, T, (g3, b3), 1e-5, True, g_mid)
            geo = dict(Ho=HW, Wo=1, T=T)
            self._gemm(bl, lambda: ops.temporal_taps(g_mid.t), P[q + "conv1"][0], hbuf, M, mode=ops.ROWS_TEMPORAL, geom=geo,
                       bias=P[q + "conv1"][1], rowbias=emb2, rb_div=HW, rb_mod=N, **self._gnkw(st_h2, HW))
            self._gn(bl, [(hbuf, cout, st_h2)], B, T * HW, T, (g4, b4), 1e-5, True, g_mid)
            # x_t = xs + conv(...);  out = alpha*xs + (1-alpha)*x_t   (util.py:358-369)
            self._gemm(bl, lambda: ops.temporal_taps(g_mid.t), P[q + "conv2"][0], out, M, mode=ops.ROWS_TEMPORAL, geom=geo,
                       bias=P[q + "conv2"][1], residual=xs, blend_x=xs, alpha=P[n + "alpha"], **self._gnkw(out_stats, HW))
            return
        # frames sharded over ranks (SURVEY F9 / 8e): the (T,H,W) statistics need the (sum, sumsq) of every rank, the GN
        # output goes into a haloed [B, T+2, HW, C] buffer whose halo frames come from the neighbour ranks, and the 3-tap
        # conv reads the haloed source.
        gh = A.want("ghalo", B * (T + 2) * HW, cout)
        geo = dict(Ho=HW, Wo=1, T=T, Tin=T + 2, t_off=1)
        r, R = self.rank, self.world
        for src, sst, (gg, bb), wkey, dst, extra in (
                (xs, st_xs, (g3, b3), "conv1", hbuf, dict(rowbias=emb2, rb_div=HW, rb_mod=N, **self._gnkw(st_h2, HW))),
                (hbuf, st_h2, (g4, b4), "conv2", out, dict(residual=xs, blend_x=xs, alpha=P[n + "alpha"],
                                                           **self._gnkw(out_stats, HW)))):
            def local_sums(dst_sums, src=src, sst=sst):
                """this rank's (sum, sumsq) per (clip, group): from the producer's unit table, or a statistics pass"""
                if sst is not None:
                    return ops.groupnorm_group_sums(sst.t, cout, None, 0, self.gn_unit, B, T, dst_sums, self.det)
                return ops.groupnorm_sums(src.t, None, B, T * HW, dst_sums, ws, self.det)
            if self.peer is not None:
                # peer memory: partial sums ride on the exchange kernel (all-reduce in one launch); the halo frames are
                # stored into the neighbours' buffers by the apply kernel itself; a second exchange orders those stores
                # before the conv (and, with the first, protects the single ghalo buffer from the next writer)
                pg = self.peer
                self._call(bl, lambda ls=local_sums: ls(self.gn_sums_local), kind="groupnorm",
                           bytes=0.0 if sst is not None else 2.0 * M * cout)
                self._call(bl, lambda: pg.exchange(self.gn_sums_local, self.gn_sums), kind="exchange")

                def apply(src=src, gg=gg, bb=bb):
                    sb = A.peers("ghalo")
                    return ops.groupnorm_apply(src.t, None, B, T * HW, self.gn_sums, self.Tg * HW, gg, bb, 1e-5, True, gh.t,
                                               (T + 2) * HW, HW, y_prev=sb.peer(r - 1), y_next=sb.peer(r + 1) if r + 1 < R else None,
                                               frame_rows=HW)
                self._call(bl, apply, kind="groupnorm", bytes=4.0 * M * cout)
                self._call(bl, lambda: pg.exchange(), kind="exchange")
            else:
                from . import dist as D
                self._call(bl, lambda ls=local_sums: ls(self.gn_sums), kind="groupnorm",
                           bytes=0.0 if sst is not None else 2.0 * M * cout)
                self._call(bl, lambda: D.allreduce_sum_(self.gn_sums, deterministic=self.det), kind="nccl")
                self._call(bl, lambda src=src, gg=gg, bb=bb: ops.groupnorm_apply(
                    src.t, None, B, T * HW, self.gn_sums, self.Tg * HW, gg, bb, 1e-5, True, gh.t, (T + 2) * HW, HW),
                    kind="groupnorm", bytes=4.0 * M * cout)
                self._call(bl, lambda: D.halo_exchange_(gh.t.view(B, T + 2, HW * cout), r, R), kind="nccl")
            self._gemm(bl, lambda: ops.temporal_taps(gh.t), P[q + wkey][0], dst, M, mode=ops.ROWS_TEMPORAL, geom=geo,
                       bias=P[q + wkey][1], **extra)

    def _transformer(self, L: Layer, xin: tuple, out: LazyBuf, out_stats, h: int, w: int):
        self._mark(L.name + "SpatialVideoTransformer")
        return self._transformer_impl(L, xin, out, out_stats, h, w)

    def _transformer_impl(self, L: Layer, xin: tuple, out: LazyBuf, out_stats, h: int, w: int):
        """SpatialVideoTransformer.forward (video_attention.py:230-301), see module docstring for the folds."""
        P, A, bl, cl, N, T, B = self.P, self.arena, self._build, self._cond_build, self.N, self.T, self.B
        x = xin[0]
        n, C = L.name, L.cin
        HW = h * w
        M = N * HW
        heads = C // self.net.cfg.num_head_channels
        if self.net.cfg.num_head_channels != 64:
            raise NotImplementedError("attention kernels are specialised for head dim 64")
        dev = self.dev
        gn, t0, t1, t2 = A.want("gn", M, C), A.want("t0", M, C), A.want("t1", M, C), A.want("t2", M, C)
        ln, qkv, att, ffh = A.want("ln", M, C), A.want("qkv", M, 3 * C), A.want("att", M, C), A.want("ffh", M, 4 * C)
        ws = self.gn_ws
        # time_pos_embed(timestep_embedding(arange(T))) : plan constant (video_attention.py:266-276)
        tpe_in = torch.zeros(T, C, dtype=F16, device=dev)
        tpe_h = torch.zeros(T, 4 * C, dtype=F16, device=dev)
        emb_t = torch.zeros(T, C, dtype=F16, device=dev)
        ops.timestep_embedding(self.frame_idx, C, tpe_in, float(self.net.cfg.max_ddpm_temb_period))
        ops.Gemm([ops.SegSpec(tpe_in)], P[n + "tpe0"][0], tpe_h, T, bias=P[n + "tpe0"][1], act=ops.ACT_SILU)()
        ops.Gemm([ops.SegSpec(tpe_h)], P[n + "tpe2"][0], emb_t, T, bias=P[n + "tpe2"][1])()

        self._gn(bl, [(x, C, xin[4])], N, HW, 1, P[n + "norm"], 1e-6, False, gn)
        self._gemm(bl, lambda: [ops.SegSpec(gn.t)], P[n + "proj_in"][0], t0, M, bias=P[n + "proj_in"][1])
        tok = t0
        for d in range(self.net.cfg.transformer_depth):
            qs, qt = n + f"transformer_blocks.{d}.", n + f"time_stack.{d}."
            # step-invariant single-token cross-attention rows (SURVEY F7): to_out(to_v(ctx)) + bias
            v_s = torch.zeros(N, C, dtype=F16, device=dev); r_s = torch.zeros(N, C, dtype=F16, device=dev)
            v_t = torch.zeros(B, C, dtype=F16, device=dev); r_t = torch.zeros(B, C, dtype=F16, device=dev)
            self._gemm(cl, lambda: [ops.SegSpec(self.ctx_in)], P[qs + "ca_v"], v_s, N)
            self._gemm(cl, lambda v_s=v_s: [ops.SegSpec(v_s)], P[qs + "ca_out"][0], r_s, N, bias=P[qs + "ca_out"][1])
            self._gemm(cl, lambda: [ops.SegSpec(self.ctx_first)], P[qt + "ca_v"], v_t, B)
            self._gemm(cl, lambda v_t=v_t: [ops.SegSpec(v_t)], P[qt + "ca_out"][0], r_t, B, bias=P[qt + "ca_out"][1])
            # ---- spatial BasicTransformerBlock (attention.py:551-572)
            self._ln(bl, tok, P[qs + "norm1"], ln, M)
            self._gemm(bl, lambda: [ops.SegSpec(ln.t)], P[qs + "qkv"], qkv, M)
            self._call(bl, lambda: ops.attention_d64(qkv.t, N, HW, heads, att.t, engine=self.attn_engine), kind="spatial_attention",
                       flops=4.0 * N * HW * HW * C, bytes=8.0 * M * C)
            self.flops += 4.0 * N * HW * HW * C
            self._gemm(bl, lambda: [ops.SegSpec(att.t)], P[qs + "to_out"][0], t1, M, bias=P[qs + "to_out"][1],
                       residual=tok, rowbias=r_s, rb_div=HW, rb_mod=N)
            self._ln(bl, t1, P[qs + "norm3"], ln, M)
            self._gemm(bl, lambda: [ops.SegSpec(ln.t)], P[qs + "ff1"][0], ffh, M, bias=P[qs + "ff1"][1], act=ops.ACT_GEGLU)
            self._gemm(bl, lambda: [ops.SegSpec(ffh.t)], P[qs + "ff2"][0], t2, M, bias=P[qs + "ff2"][1], residual=t1)
            # ---- temporal VideoTransformerBlock on x_mix = t2 + emb_t (video_attention.py:109-140, :286-289)
            self._ln(bl, t2, P[qt + "norm_in"], ln, M, addvec=emb_t, add_div=HW, add_mod=T)
            self._gemm(bl, lambda: [ops.SegSpec(ln.t)], P[qt + "ff_in1"][0], ffh, M, bias=P[qt + "ff_in1"][1],
                       act=ops.ACT_GEGLU)
            u0 = t0          # the block input `tok` is dead once attn1's output projection has consumed it
            self._gemm(bl, lambda: [ops.SegSpec(ffh.t)], P[qt + "ff_in2"][0], u0, M, bias=P[qt + "ff_in2"][1],
                       residual=t2, rowbias=emb_t, rb_div=HW, rb_mod=T)
            self._ln(bl, u0, P[qt + "norm1"], ln, M)
            self._gemm(bl, lambda: [ops.SegSpec(ln.t)], P[qt + "qkv"], qkv, M)
            if self.shard is None:
                self._call(bl, lambda: ops.temporal_attention_d64(qkv.t, B, T, HW, heads, att.t), kind="temporal_attention",
                           flops=4.0 * N * HW * T * C, bytes=8.0 * M * C)
            elif self.peer is not None:
                # pixel-strip sharding over peer memory: this rank attends pixel strip `rank` for ALL Tg frames, reading the
                # other ranks' q|k|v rows from their buffers and storing their frames' outputs into their `att` buffers
                pg = self.peer
                self._call(bl, lambda: pg.exchange(), kind="exchange")           # every rank's q|k|v is written
                self._call(bl, lambda: ops.temporal_attention_d64_sharded(A.peers("qkv"), A.peers("att"), self.rank, self.world,
                                                                          B, T, HW, heads),
                           kind="temporal_attention", flops=4.0 * N * HW * self.Tg * C, bytes=8.0 * M * C)
                self._call(bl, lambda: pg.exchange(), kind="exchange")           # every rank's `att` rows have arrived
            else:
                # NCCL form: all-gather q|k|v rows of every rank (frame order), attend over all Tg frames, keep the local frames
                from . import dist as D
                Tg, r = self.Tg, self.rank
                qkv_f, att_f = A.want("qkv_full", B * Tg * HW, 3 * C), A.want("att_full", B * Tg * HW, C)
                self._call(bl, lambda: D.gather_frames_(qkv.t, qkv_f.t, B, T * HW, self.world), kind="nccl")
                self._call(bl, lambda: ops.temporal_attention_d64(qkv_f.t, B, Tg, HW, heads, att_f.t),
                           kind="temporal_attention", flops=4.0 * B * Tg * HW * Tg * C, bytes=8.0 * B * Tg * HW * C)

                def keep_local(att=att, att_f=att_f):
                    for b in range(B):
                        att.t[b * T * HW:(b + 1) * T * HW].copy_(att_f.t[(b * Tg + r * T) * HW:(b * Tg + (r + 1) * T) * HW])
                self._call(bl, keep_local, kind="copy")
            self.flops += 4.0 * N * HW * T * C
            self._gemm(bl, lambda: [ops.SegSpec(att.t)], P[qt + "to_out"][0], t1, M, bias=P[qt + "to_out"][1],
                       residual=u0, rowbias=r_t, rb_div=T * HW, rb_mod=B)
            self._ln(bl, t1, P[qt + "norm3"], ln, M)
            self._gemm(bl, lambda: [ops.SegSpec(ln.t)], P[qt + "ff1"][0], ffh, M, bias=P[qt + "ff1"][1], act=ops.ACT_GEGLU)
            # x = alpha * x_spatial + (1 - alpha) * x_mix      (video_attention.py:290-294)
            self._gemm(bl, lambda: [ops.SegSpec(ffh.t)], P[qt + "ff2"][0], t0, M, bias=P[qt + "ff2"][1], residual=t1,
                       blend_x=t2, alpha=P[n + "alpha"])
            tok = t0
        self._gemm(bl, lambda: [ops.SegSpec(tok.t)], P[n + "proj_out"][0], out, M, bias=P[n + "proj_out"][1], residual=x,
                   **self._gnkw(out_stats, HW))

    def _ln(self, lst, x: LazyBuf, gb, y: LazyBuf, M, addvec=None, add_div=1, add_mod=1):
        g, b = gb
        self._call(lst, lambda: ops.layernorm(x.t, g, b, y.t, M, addvec=addvec, add_div=add_div, add_mod=add_mod),
                   kind="layernorm", bytes=4.0 * M * x.cols)

    # ---- per-video / per-step entry points ------------------------------------------------------------------------
    def prepare_conditioning(self, context: torch.Tensor, y: torch.Tensor):
        """context (N|B, 1, ctx) and y (N|B, adm): label_emb(y) and the single-token cross-attention rows."""
        N, T, B = self.N, self.T, self.B
        if context.dim() != 3 or context.shape[1] != 1:
            raise NotImplementedError(f"context of shape {tuple(context.shape)}: the Hi3D path has exactly one "
                                      f"conditioning token (SURVEY F7); multi-token cross-attention is not built")
        ctx = context[:, 0]
        if ctx.shape[0] == B and B != N:
            ctx = ctx.repeat_interleave(T, dim=0)         # video_model.py:463-465
        if y.shape[0] == B and B != N:
            y = y.repeat_interleave(T, dim=0)             # video_model.py:460-462
        assert ctx.shape[0] == N and y.shape[0] == N
        self.ctx_in.copy_(ctx)
        self.ctx_first.copy_(ctx[::T])                    # video_attention.py:250
        self.y_in.copy_(y)
        for s in self.cond_steps:
            s()

    def set_timesteps(self, t: torch.Tensor):
        self.t_in.copy_(t.reshape(-1).float())

    def run(self):
        for s in self.steps:
            s()
        if self._nvtx_open:
            torch.cuda.nvtx.range_pop()
            self._nvtx_open = False

    def launches_per_step(self) -> int:
        from . import _native
        a = _native.launch_count()
        self.run()
        return _native.launch_count() - a
