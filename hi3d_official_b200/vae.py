"""AutoencoderKL (2-D, per frame): drop-in for `sgm.models.autoencoder.AutoencoderKL` /
`AutoencoderKLModeOnly` (autoencoder.py:436-520,606-619) with the Encoder / Decoder of
sgm/modules/diffusionmodules/model.py:487-748 compiled into a flat launch plan of the same C-ABI kernels as
the UNet: GN(eps 1e-6)+swish -> implicit-GEMM conv3x3 (nin_shortcut folded in as extra K segments),
asymmetric-pad stride-2 down conv, nearest-x2 fused into the up conv's gather, and the single-head d=512 mid
attention as two GEMMs around a row softmax.  State-dict keys/shapes are the reference's.

`encode(x)` / `decode(z)` take and return NCHW tensors like the reference; all compute is fp16 with fp32
accumulation (the reference runs the first stage in pure fp16: `disable_first_stage_autocast`, SURVEY F5).
"""
from __future__ import annotations

import os

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import ops, pack
from .spec import VAEConfig, vae_param_shapes
from .unet import Arena, LazyBuf, StatsBuf, _ParamTree

F16 = torch.float16
CIN_PAD = 64
COUT_PAD = 8


class _VAEPlan:
    """Launch plan for encoder or decoder at one (n, H, W)."""

    def __init__(self, ae: "AutoencoderKL", which: str, n: int, H: int, W: int, T: int = 0, det: bool = False):
        self.ae, self.which, self.n, self.H, self.W, self.T = ae, which, n, H, W, T
        self.det = det                 # deterministic GroupNorm statistics (ops.deterministic())
        self._part_floats = 0          # deterministic mode: partials scratch shared by every statistics producer
        self.gn_part = None
        self.P = ae._pack()
        self.dev = ae.device
        self.A = Arena(self.dev)
        self._build: List = []
        self.flops = 0.0
        self.gn_ws = ops.groupnorm_ws(n, self.dev)
        self._pp = 0
        # GroupNorm statistics from the producing GEMM epilogues (hi3d_gemm_params::gn_stats), as in the UNet plan
        self.gn_unit = max(1, ae.cfg.ch // 32)
        self.gn_fused = (os.environ.get("HI3D_GN_FUSED", "1") != "0" and ae.cfg.ch % 32 == 0
                         and ae.cfg.ch * max(ae.cfg.ch_mult) // self.gn_unit <= 256)
        self._stats_floats = 0
        self.stats_arena = None
        self._last_stats = {}          # id(LazyBuf) -> StatsBuf of the tensor it currently holds
        if self.gn_fused:
            self._call(lambda: self.stats_arena.zero_())
        if which == "enc":
            self._compile_encoder()
        elif which == "vdec":
            self._compile_decoder(video=True)
        else:
            self._compile_decoder()
        self.A.materialise()
        if self.gn_fused:
            self.stats_arena = torch.zeros(max(self._stats_floats, 2), dtype=torch.float32, device=self.dev)
        if self.det:
            self.gn_part = torch.empty(max(self._part_floats, 4), dtype=torch.float32, device=self.dev)
        self.steps = [b() for b in self._build]
        self._build = None

    # -- emit helpers ------------------------------------------------------------------------------------------
    def _gemm(self, segs_fn, W, out, M, **kw):
        def build():
            def res(v):
                return v.t if isinstance(v, (LazyBuf, StatsBuf)) else (v() if callable(v) else v)
            k2 = {k: res(v) for k, v in kw.items()}
            if self.det and "gn_stats" in k2:
                k2["gn_partials"] = self.gn_part
            g = ops.Gemm(segs_fn(), res(W), res(out), M, engine=self.ae.engine, **k2)
            self.flops += g.flops
            return g
        self._build.append(build)

    def _call(self, fn):
        self._build.append(lambda: fn)

    def _track(self, out: LazyBuf, C: int, rows_per_img: int) -> dict:
        """Gemm kwargs: the epilogue accumulates the GroupNorm statistics of `out` (consumed by the next _gn on it)."""
        if not self.gn_fused or C % 32 or C % self.gn_unit or C // self.gn_unit > 256:      # (C % 32: never a GroupNorm input)
            self._last_stats.pop((out.tag, out.rows, out.cols), None)
            return {}
        sb = StatsBuf(self, self._stats_floats, self.n, C // self.gn_unit)
        self._stats_floats += self.n * (C // self.gn_unit) * 2
        self._last_stats[(out.tag, out.rows, out.cols)] = sb
        if self.det:
            self._part_floats = max(self._part_floats, ops.groupnorm_partials_floats(self.n, out.rows // self.n, C, self.gn_unit))
        return dict(gn_stats=sb, gn_unit=self.gn_unit, gn_rows=rows_per_img)

    def _nxt(self, rows, C):
        self._pp ^= 1
        return self.A.want(f"blk{self._pp}", rows, C)

    def _gn(self, x: LazyBuf, key: str, rows_per_img: int, y: LazyBuf, silu=True, eps=1e-6, ips=1):
        """GroupNorm(32)[+swish]; ips = images per sample (T for the (T,H,W) statistics of a time_stack)."""
        g, b = self.P[key]
        st = self._last_stats.get((x.tag, x.rows, x.cols))
        ns, rows = self.n // ips, rows_per_img * ips
        if st is not None:
            self._call(lambda: ops.groupnorm_apply_stats(x.t, st.t, None, None, self.gn_unit, ns, rows, ips, rows, g, b, eps,
                                                         silu, y.t))
        else:
            self._call(lambda: ops.groupnorm_silu(x.t, None, ns, rows, g, b, eps, silu, y.t, self.gn_ws, self.det))

    def _conv(self, src: LazyBuf, key: str, out: LazyBuf, ho, wo, hs, ws, stride=1, ups=0, pad_lo=1, **kw):
        Wt, b = self.P[key]
        self._gemm(lambda: ops.conv_taps([src.t], pad_lo=pad_lo), Wt, out, self.n * ho * wo, mode=ops.ROWS_CONV2D,
                   geom=dict(Ho=ho, Wo=wo, Hs=hs, Ws=ws, stride=stride, ups=ups), bias=b, **self._track(out, out.cols, ho * wo),
                   **kw)

    def _resnet(self, pre: str, x: LazyBuf, cin: int, cout: int, h: int, w: int) -> LazyBuf:
        """ResnetBlock.forward, model.py:131-151 (temb is None)."""
        M = self.n * h * w
        g1, hb, g2 = self.A.want("gn", M, cin), self.A.want("h", M, cout), self.A.want("gn", M, cout)
        out = self._nxt(M, cout)
        self._gn(x, pre + "norm1", h * w, g1)
        self._conv(g1, pre + "conv1", hb, h, w, h, w)
        self._gn(hb, pre + "norm2", h * w, g2)
        Wt, b = self.P[pre + "conv2"]
        geo = dict(Ho=h, Wo=w, Hs=h, Ws=w)
        if cin != cout:    # nin_shortcut 1x1 as one more K segment over the raw input
            self._gemm(lambda: ops.conv_taps([g2.t]) + [ops.SegSpec(x.t)], Wt, out, M, mode=ops.ROWS_CONV2D, geom=geo,
                       bias=b, **self._track(out, cout, h * w))
        else:
            self._gemm(lambda: ops.conv_taps([g2.t]), Wt, out, M, mode=ops.ROWS_CONV2D, geom=geo, bias=b, residual=x,
                       **self._track(out, cout, h * w))
        return out

    def _video_resnet(self, pre: str, x: LazyBuf, cin: int, cout: int, h: int, w: int) -> LazyBuf:
        """temporal_ae.VideoResBlock.forward (temporal_ae.py:62-81): the spatial ResnetBlock, then the `time_stack`
        ResBlock(dims=3, kernel (3,1,1), no emb; openaimodel.py:328-354) on the (b, c, t, h, w) view -- GroupNorm over
        (C/32, T, H, W), eps 1e-5 -- and x = a * time_stack(x) + (1 - a) * x with a = sigmoid(mix_factor): NOTE the blend
        weighs the TEMPORAL branch (the UNet's AlphaBlender weighs the spatial one).  time_stack(x) = x + h, so
        out = x + a h = (1 - a) x + a (x + h): the engine's blend epilogue with alpha_engine = 1 - a."""
        xs = self._resnet(pre, x, cin, cout, h, w)
        T, n = self.T, self.n
        B, HW = n // T, h * w
        M = n * HW
        A = self.A
        g, hb = A.want("gn", M, cout), A.want("h", M, cout)
        out = self._nxt(M, cout)
        q = pre + "time_stack."
        geo = dict(Ho=HW, Wo=1, T=T)
        a = self.P[pre + "mix_factor"]

        self._gn(xs, q + "in_layers.0", HW, g, eps=1e-5, ips=T)
        W1, b1 = self.P[q + "in_layers.2"]
        self._gemm(lambda: ops.temporal_taps(g.t), W1, hb, M, mode=ops.ROWS_TEMPORAL, geom=geo, bias=b1,
                   **self._track(hb, cout, HW))
        self._gn(hb, q + "out_layers.0", HW, g, eps=1e-5, ips=T)
        W2, b2 = self.P[q + "out_layers.3"]
        self._gemm(lambda: ops.temporal_taps(g.t), W2, out, M, mode=ops.ROWS_TEMPORAL, geom=geo, bias=b2, residual=xs,
                   blend_x=xs, alpha=1.0 - a, **self._track(out, cout, HW))
        return out

    def _attn(self, pre: str, x: LazyBuf, C: int, h: int, w: int) -> LazyBuf:
        """AttnBlock.forward, model.py:180-201: one head, d = C, softmax(q k^T * C^-0.5) v per image, as
        scores = GEMM(q, k) -> row softmax -> GEMM(P, v^T) on the same engine as everything else."""
        n, L = self.n, h * w
        M = n * L
        A = self.A
        if C == 512 and L % 128 == 0 and self.ae.engine == "tc5":
            # flash attention on tcgen05: q|k|v as ONE GEMM, fp32 scores / softmax inside the kernel, no L x L buffer
            g, qkv, o = A.want("gn", M, C), A.want("qkv", M, 3 * C), A.want("att", M, C)
            out = self._nxt(M, C)
            self._gn(x, pre + "norm", L, g, silu=False)
            Wq, bq = self.P[pre + "qkv"]
            self._gemm(lambda: [ops.SegSpec(g.t)], Wq, qkv, M, bias=bq)
            self._call(lambda: ops.attention_d512(qkv.t, n, L, o.t, float(C) ** -0.5))
            Wo, bo = self.P[pre + "proj_out"]
            self._gemm(lambda: [ops.SegSpec(o.t)], Wo, out, M, bias=bo, residual=x, **self._track(out, C, L))
            return out
        # small / odd sizes (L not a multiple of 128) and the mma.sync engine: scores through the GEMM engine, one image at a
        # time (an L x L fp16 buffer of SCALED logits -- fine for the tiny test shapes this path still serves)
        if L % 64:
            raise NotImplementedError(f"VAE attention needs (H/8)*(W/8) % 64 == 0, got {L}")
        g, q, k, v, o = (A.want(t, M, C) for t in ("gn", "q", "k", "v", "att"))
        S, vt = A.want("scores", L, L), A.want("vt", C, L)
        out = self._nxt(M, C)
        self._gn(x, pre + "norm", L, g, silu=False)
        for nm, dst in (("q_scaled", q), ("k", k), ("v", v)):
            Wt, b = self.P[pre + nm]
            self._gemm(lambda: [ops.SegSpec(g.t)], Wt, dst, M, bias=b)
        for i in range(n):
            sl = slice(i * L, (i + 1) * L)
            self._call(lambda sl=sl: ops.transpose(v.t[sl], L, C, C, vt.t))
            self._gemm(lambda sl=sl: [ops.SegSpec(q.t[sl])], lambda sl=sl: k.t[sl], S, L)
            self._call(lambda: ops.softmax_rows(S.t, L, L, 1.0))
            self._gemm(lambda: [ops.SegSpec(S.t)], vt, lambda sl=sl: o.t[sl], L)
        Wo, bo = self.P[pre + "proj_out"]
        self._gemm(lambda: [ops.SegSpec(o.t)], Wo, out, M, bias=bo, residual=x, **self._track(out, C, L))
        return out

    # -- encoder / decoder walks ----------------------------------------------------------------------------------
    def _compile_encoder(self):
        """Encoder.forward, model.py:576-601 + quant_conv (autoencoder.py:470-471)."""
        cfg, n, H, W, A = self.ae.cfg, self.n, self.H, self.W, self.A
        nres = len(cfg.ch_mult)
        if H % (1 << (nres - 1)) or W % (1 << (nres - 1)):
            raise ValueError(f"image size {H}x{W} must be divisible by {1 << (nres - 1)}")
        self.xin = A.want("xin", n * H * W, CIN_PAD)
        h, w = H, W
        cur = self._nxt(n * h * w, cfg.ch)
        self._conv(self.xin, "encoder.conv_in", cur, h, w, h, w)
        in_mult = (1,) + tuple(cfg.ch_mult)
        bi = cfg.ch
        for lvl in range(nres):
            bi, bo = cfg.ch * in_mult[lvl], cfg.ch * cfg.ch_mult[lvl]
            for b in range(cfg.num_res_blocks):
                cur = self._resnet(f"encoder.down.{lvl}.block.{b}.", cur, bi, bo, h, w)
                bi = bo
            if lvl != nres - 1:   # Downsample: F.pad (0,1,0,1) + conv3x3 stride 2 pad 0 (model.py:84-88)
                out = self._nxt(n * (h // 2) * (w // 2), bi)
                self._conv(cur, f"encoder.down.{lvl}.downsample.conv", out, h // 2, w // 2, h, w, stride=2, pad_lo=0)
                cur, h, w = out, h // 2, w // 2
        cur = self._resnet("encoder.mid.block_1.", cur, bi, bi, h, w)
        cur = self._attn("encoder.mid.attn_1.", cur, bi, h, w)
        cur = self._resnet("encoder.mid.block_2.", cur, bi, bi, h, w)
        M = n * h * w
        g = A.want("gn", M, bi)
        self._gn(cur, "encoder.norm_out", h * w, g)
        mom = A.want("h", M, 64)     # conv_out output, padded to 64 channels so quant_conv (1x1) sees one K segment
        self._conv(g, "encoder.conv_out", mom, h, w, h, w)
        self.out = A.want("moments", M, COUT_PAD)
        Wq, bq = self.P["quant_conv"]
        self._gemm(lambda: [ops.SegSpec(mom.t)], Wq, self.out, M, bias=bq)
        self.out_hw = (h, w)

    def _compile_decoder(self, video: bool = False):
        """post_quant_conv (autoencoder.py:492) + Decoder.forward, model.py:715-748.  (H, W) are LATENT dims.
        video=True: temporal_ae.VideoDecoder (time_mode 'conv-only', temporal_ae.py:293-349) run as
        Decoder.forward(z, timesteps=T): VideoResBlocks instead of ResnetBlocks, plain AttnBlock, AE3DConv as conv_out."""
        cfg, n, h, w, A = self.ae.cfg, self.n, self.H, self.W, self.A
        if video and (self.T <= 0 or n % self.T):
            raise ValueError(f"VideoDecoder: batch {n} is not a multiple of timesteps {self.T}")
        resnet = self._video_resnet if video else self._resnet
        nres = len(cfg.ch_mult)
        self.xin = A.want("xin", n * h * w, CIN_PAD)
        zq = A.want("h", n * h * w, CIN_PAD)
        Wp, bp = self.P["post_quant_conv"]
        self._gemm(lambda: [ops.SegSpec(self.xin.t)], Wp, zq, n * h * w, bias=bp)
        bi = cfg.ch * cfg.ch_mult[-1]
        cur = self._nxt(n * h * w, bi)
        self._conv(zq, "decoder.conv_in", cur, h, w, h, w)
        cur = resnet("decoder.mid.block_1.", cur, bi, bi, h, w)
        cur = self._attn("decoder.mid.attn_1.", cur, bi, h, w)
        cur = resnet("decoder.mid.block_2.", cur, bi, bi, h, w)
        for lvl in reversed(range(nres)):
            bo = cfg.ch * cfg.ch_mult[lvl]
            for b in range(cfg.num_res_blocks + 1):
                cur = resnet(f"decoder.up.{lvl}.block.{b}.", cur, bi, bo, h, w)
                bi = bo
            if lvl != 0:          # Upsample: nearest x2 + conv3x3 (model.py:67-71), fused into the gather
                out = self._nxt(n * 4 * h * w, bi)
                parity, ub = self.P[f"decoder.up.{lvl}.upsample.conv"]
                trk = self._track(out, bi, h * w)               # one statistics table for the four parity launches
                for (py, px), (Wt, shifts) in parity.items():   # nearest-x2 + conv3x3 == 4 parity-class 2x2 convs
                    self._gemm(lambda shifts=shifts, cur=cur: [ops.SegSpec(cur.t, dy=sy, dx=sx) for sy, sx in shifts], Wt,
                               out, n * h * w, mode=ops.ROWS_CONV2D,
                               geom=dict(Ho=h, Wo=w, Hs=h, Ws=w, out_up=1, out_py=py, out_px=px), bias=ub, **trk)
                cur, h, w = out, 2 * h, 2 * w
        M = n * h * w
        g = A.want("gn", M, bi)
        self._gn(cur, "decoder.norm_out", h * w, g)
        self.out = A.want("img", M, COUT_PAD)
        if not video:
            self._conv(g, "decoder.conv_out", self.out, h, w, h, w)
        else:
            # AE3DConv (temporal_ae.py:84-108): the 2-D conv (output padded to one 64-wide K segment), then the Conv3d
            # (3,1,1) over the frames of the (b, c, t, h, w) view as a frame-tap GEMM
            mid = A.want("h", M, CIN_PAD)
            self._conv(g, "decoder.conv_out", mid, h, w, h, w)
            Wt, bt = self.P["decoder.conv_out.time_mix_conv"]
            self._gemm(lambda: ops.temporal_taps(mid.t), Wt, self.out, M, mode=ops.ROWS_TEMPORAL,
                       geom=dict(Ho=h * w, Wo=1, T=self.T), bias=bt)
        self.out_hw = (h, w)

    def run(self):
        for s in self.steps:
            s()


class _Net(nn.Module):
    """Parameter holder exposing `.encoder` / `.decoder` style attribute access for isinstance-free callers."""


class Encoder(_ParamTree):
    pass


class Decoder(_ParamTree):
    pass


class AutoencoderKL(nn.Module):
    """sgm.models.autoencoder.AutoencoderKL: `embed_dim`, `ddconfig` (+ ignored training kwargs such as
    lossconfig / monitor / ckpt_path=None).  regularizer = DiagonalGaussianRegularizer(sample=True)."""
    sample_posterior = True

    def __init__(self, embed_dim: int = 4, ddconfig: Optional[dict] = None, **ignored):
        super().__init__()
        if ddconfig is None:
            raise ValueError("ddconfig is required")
        if ignored.get("ckpt_path") is not None:
            raise NotImplementedError("ckpt_path in the first-stage config: load weights with load_state_dict")
        self.cfg = VAEConfig.from_ddconfig(ddconfig, embed_dim)
        self.embed_dim = embed_dim
        self.encoder, self.decoder = Encoder(), self._make_decoder()
        self.quant_conv, self.post_quant_conv = _ParamTree(), _ParamTree()
        roots = {"encoder": self.encoder, "decoder": self.decoder, "quant_conv": self.quant_conv,
                 "post_quant_conv": self.post_quant_conv}
        for name, shp in self._param_shapes(ignored).items():
            root, rest = name.split(".", 1)
            roots[root].put(rest, nn.Parameter(torch.empty(shp), requires_grad=False))
        self._packed = None
        self._plans: Dict[tuple, _VAEPlan] = {}
        self.engine = os.environ.get("HI3D_ENGINE", "tc5")     # "tc5" = tcgen05/TMEM/TMA engine, "mma" = mma.sync engine
        self.max_batch_size = ignored.get("max_batch_size", None)
        # a parent's load_state_dict (DiffusionEngine.init_from_ckpt) recurses through _load_from_state_dict and never
        # reaches the override below: invalidate the packed weights / plans from a pre-hook as well
        self._register_load_state_dict_pre_hook(lambda *a, **k: self._invalidate())

    def _param_shapes(self, kwargs: dict):
        return vae_param_shapes(self.cfg)

    def _make_decoder(self):
        return Decoder()

    # -- lifecycle ----------------------------------------------------------------------------------------------------
    def _invalidate(self):
        self._packed, self._plans = None, {}

    def _apply(self, fn, *a, **k):
        self._invalidate()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._invalidate()
        return super().load_state_dict(*a, **k)

    def set_engine(self, engine: str):
        if engine != self.engine:
            self.engine, self._plans = engine, {}

    @property
    def device(self):
        return self.quant_conv.weight.device

    def _pack(self) -> dict:
        if self._packed is not None:
            return self._packed
        if self.device.type != "cuda":
            raise RuntimeError("hi3d_official_b200.AutoencoderKL computes only on CUDA; there is no CPU fallback")
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        P = {}
        temporal = isinstance(self.decoder, VideoDecoder)
        for k in sd:
            if k.endswith("mix_factor"):                       # temporal_ae.VideoResBlock: alpha = sigmoid(mix_factor)
                P[k] = float(torch.sigmoid(sd[k].float()).item())
                continue
            if not k.endswith(".weight"):
                continue
            base = k[:-7]
            w, b = sd[k], sd[base + ".bias"]
            if w.dim() == 1:                                   # GroupNorm affine
                P[base] = (w.float().contiguous(), b.float().contiguous())
            elif base == "decoder.conv_out.time_mix_conv":     # AE3DConv's Conv3d (3,1,1) on out_ch channels
                P[base] = (pack.pack_conv3d_t(w, cin_pad=CIN_PAD, cout_pad=COUT_PAD), pack.pack_bias(b, w.shape[0], COUT_PAD))
            elif w.dim() == 5:                                 # time_stack convs (Co, Ci, 3, 1, 1)
                P[base] = (pack.pack_conv3d_t(w), b.float().contiguous())
            elif base == "decoder.conv_out" and temporal:      # feeds time_mix_conv: one 64-wide K segment per frame tap
                P[base] = (pack.pack_conv2d(w, cout_pad=CIN_PAD), pack.pack_bias(b, w.shape[0], CIN_PAD))
            elif base.endswith("nin_shortcut"):
                continue                                       # folded into conv2 below
            elif base in ("encoder.conv_in",):
                P[base] = (pack.pack_conv2d(w, cin_pad=CIN_PAD), b.float().contiguous())
            elif base == "decoder.conv_in":
                P[base] = (pack.pack_conv2d(w, cin_pad=CIN_PAD), b.float().contiguous())
            elif base == "encoder.conv_out":                   # 2*z channels -> padded to 64 (feeds quant_conv)
                P[base] = (pack.pack_conv2d(w, cout_pad=64), pack.pack_bias(b, w.shape[0], 64))
            elif base.endswith("upsample.conv"):
                P[base] = (pack.pack_upconv_parity(w), b.float().contiguous())
            elif base == "decoder.conv_out":
                P[base] = (pack.pack_conv2d(w, cout_pad=COUT_PAD), pack.pack_bias(b, w.shape[0], COUT_PAD))
            elif base == "quant_conv":                         # 1x1: K padded to 64, N padded to 8
                P[base] = (pack.pack_conv2d(w, cin_pad=64, cout_pad=COUT_PAD), pack.pack_bias(b, w.shape[0], COUT_PAD))
            elif base == "post_quant_conv":                    # 1x1: K padded to 64, N padded to 64 (feeds conv_in)
                P[base] = (pack.pack_conv2d(w, cin_pad=CIN_PAD, cout_pad=CIN_PAD), pack.pack_bias(b, w.shape[0], CIN_PAD))
            elif base.endswith("conv2") and (base[:-5] + "nin_shortcut.weight") in sd:
                ws_, bs_ = sd[base[:-5] + "nin_shortcut.weight"], sd[base[:-5] + "nin_shortcut.bias"]
                P[base] = (pack.cat_k(pack.pack_conv2d(w), pack.pack_conv2d(ws_)), (b.float() + bs_.float()).contiguous())
            else:
                P[base] = (pack.pack_conv2d(w), b.float().contiguous())
        for pre in ("encoder.mid.attn_1.", "decoder.mid.attn_1."):      # q | k | v of the AttnBlock as one [3C, C] GEMM
            if pre + "q" in P:
                P[pre + "qkv"] = (torch.cat([P[pre + n_][0] for n_ in "qkv"], 0).contiguous(),
                                  torch.cat([P[pre + n_][1] for n_ in "qkv"], 0).contiguous())
                # GEMM-softmax-GEMM fallback (L % 128 != 0): its L x L score buffer is fp16, so the softmax scale
                # C^-0.5 is folded into the q projection -- the stored logits are the scaled ones, as in the reference
                Wq_, bq_ = P[pre + "q"]
                sc = float(Wq_.shape[0]) ** -0.5
                P[pre + "q_scaled"] = ((Wq_.float() * sc).to(Wq_.dtype).contiguous(), (bq_ * sc).contiguous())
        self._packed = P
        return P

    def _plan(self, which: str, n: int, H: int, W: int, T: int = 0) -> _VAEPlan:
        key = (which, n, H, W, self.engine, T, ops.deterministic())
        if key not in self._plans:
            self._plans[key] = _VAEPlan(self, which, n, H, W, T, det=key[-1])
        return self._plans[key]

    # -- reference API --------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def encode_moments(self, x: torch.Tensor) -> Tuple[torch.Tensor, Tuple[int, int]]:
        n, c, H, W = x.shape
        plan = self._plan("enc", n, H, W)
        ops.nchw_to_nhwc(x.contiguous(), plan.xin.t.view(n, H, W, CIN_PAD))
        plan.run()
        return plan.out.t, plan.out_hw

    @torch.no_grad()
    def encode(self, x: torch.Tensor, return_reg_log: bool = False, noise: Optional[torch.Tensor] = None,
               scale: float = 1.0):
        """autoencoder.py:468-488.  Posterior sampling draws CPU randn exactly like the reference
        (distributions.py:37-41) unless `noise` is supplied; AutoencoderKLModeOnly returns the mode."""
        if x.dtype not in (torch.float16, torch.float32):
            x = x.float()
        bs = self.max_batch_size or x.shape[0]
        outs = []
        for i in range(0, x.shape[0], bs):
            xb = x[i:i + bs]
            mom, (h, w) = self.encode_moments(xb)
            z = torch.empty(xb.shape[0], self.embed_dim, h, w, dtype=torch.float32, device=x.device)
            nz = None
            if self.sample_posterior:
                nz = noise[i:i + bs] if noise is not None else torch.randn(z.shape).to(device=x.device)
                nz = nz.float().contiguous()
            ops.gaussian_sample(mom, nz, z, scale)
            outs.append(z)
        z = torch.cat(outs, 0) if len(outs) > 1 else outs[0]
        z = z.to(x.dtype)
        return (z, {}) if return_reg_log else z

    @torch.no_grad()
    def decode(self, z: torch.Tensor, scale: float = 1.0, **decoder_kwargs) -> torch.Tensor:
        """autoencoder.py:490-505 (post_quant_conv + decoder); returns NCHW in z's dtype."""
        temporal = isinstance(self.decoder, VideoDecoder)
        T = int(decoder_kwargs.pop("timesteps", 0)) if temporal else 0
        if decoder_kwargs:
            raise NotImplementedError(f"decoder kwargs {list(decoder_kwargs)}: the 2-D decoder takes none; the temporal "
                                      f"decoder (AutoencoderKLTemporal) takes timesteps=T")
        if temporal and T <= 0:
            raise ValueError("the temporal decoder needs decode(z, timesteps=T) (diffusion.py:126-129)")
        if z.dtype not in (torch.float16, torch.float32):
            z = z.float()
        bs = self.max_batch_size or z.shape[0]
        if temporal:                      # whole clips per launch plan
            bs = max(T, bs // T * T)
        outs = []
        for i in range(0, z.shape[0], bs):
            zb = z[i:i + bs].contiguous()
            n, c, h, w = zb.shape
            plan = self._plan("vdec", n, h, w, T) if temporal else self._plan("dec", n, h, w)
            ops.nchw_to_nhwc(zb, plan.xin.t.view(n, h, w, CIN_PAD), scale)
            plan.run()
            H, W = plan.out_hw
            img = torch.empty(n, self.cfg.out_ch, H, W, dtype=z.dtype, device=z.device)
            ops.nhwc_to_nchw(plan.out.t, img)
            outs.append(img)
        return torch.cat(outs, 0) if len(outs) > 1 else outs[0]

    def forward(self, x: torch.Tensor, **kw):
        z = self.encode(x)
        return z, self.decode(z), {}


class VideoDecoder(Decoder):
    """Parameter tree of sgm.modules.autoencoding.temporal_ae.VideoDecoder (temporal_ae.py:293-349).  Its presence as
    `first_stage_model.decoder` is what makes DiffusionEngine.decode_first_stage pass timesteps (diffusion.py:126-129)."""


class AutoencoderKLTemporal(AutoencoderKL):
    """The temporal first stage north_star calls "AutoencoderKLTemporal" (SURVEY F3 / §8f N1): the 2-D Encoder with the
    temporal `VideoDecoder` of sgm/modules/autoencoding/temporal_ae.py (as in SVD's AutoencodingEngine config): every
    ResnetBlock is a VideoResBlock (spatial block + (3,1,1) time_stack ResBlock + learned blend), conv_out is an AE3DConv;
    `time_mode` 'conv-only' (plain AttnBlock), `video_kernel_size` [3, 1, 1].  decode(z, timesteps=T).
    State-dict keys / shapes: spec.video_decoder_param_shapes (checked against the unmodified reference class)."""

    def _param_shapes(self, kwargs: dict):
        from .spec import video_decoder_param_shapes
        vks = kwargs.get("video_kernel_size", [3, 1, 1])
        k3 = tuple(vks) if not isinstance(vks, int) else (vks,) * 3
        if k3 != (3, 1, 1):
            raise NotImplementedError(f"video_kernel_size {vks}: only [3, 1, 1] (frame taps) is built; spatially extended "
                                      f"temporal kernels would need (dt, dy, dx) taps in the implicit-GEMM engine")
        if kwargs.get("time_mode", "conv-only") != "conv-only":
            raise NotImplementedError("time_mode other than 'conv-only' (temporal attention inside the VAE) is not built")
        shapes = vae_param_shapes(self.cfg)
        out = type(shapes)((k, v) for k, v in shapes.items() if not k.startswith("decoder."))
        out.update(video_decoder_param_shapes(self.cfg, k3))
        return out

    def _make_decoder(self):
        return VideoDecoder()


class AutoencoderKLModeOnly(AutoencoderKL):
    """autoencoder.py:606-619: DiagonalGaussianRegularizer(sample=False)."""
    sample_posterior = False
