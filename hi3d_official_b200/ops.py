"""Thin typed wrappers that turn torch CUDA tensors into C-ABI calls (pointers + sizes + stream).

torch is used for device memory and streams only; every function here ends in exactly one
`libhi3d_b200.so` entry point and raises if that fails.  `Gemm` pre-bakes its parameter block once so a
replayed step costs one ctypes call per launch.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import torch

from . import _native as N
from ._native import ACT_GEGLU, ACT_NONE, ACT_SILU, ROWS_CONV2D, ROWS_PLAIN, ROWS_TEMPORAL  # noqa: F401

F16 = torch.float16


def deterministic() -> bool:
    """The deterministic-mode switch, read when a launch plan is built (and part of its key): GroupNorm statistics without
    float atomics, so that the same inputs give bit-identical outputs.  On with torch.use_deterministic_algorithms(True) or
    HI3D_DETERMINISTIC=1 (for jobs that cannot change code, e.g. torchrun / bench.py)."""
    return torch.are_deterministic_algorithms_enabled() or os.environ.get("HI3D_DETERMINISTIC") == "1"


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _chk16(t: torch.Tensor, name: str):
    if t.dtype != F16 or not t.is_cuda or not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous CUDA fp16 tensor, got {t.dtype} {t.device} "
                         f"contiguous={t.is_contiguous()}")


def _chk32(t: torch.Tensor, name: str):
    if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous CUDA fp32 tensor")


class SegSpec:
    """One K-segment of the implicit-GEMM A operand (see hi3d_seg)."""
    __slots__ = ("src", "ld", "c_off", "C", "dy", "dx", "dt")

    def __init__(self, src: torch.Tensor, C_: Optional[int] = None, c_off: int = 0, dy: int = 0, dx: int = 0,
                 dt: int = 0, ld: Optional[int] = None):
        _chk16(src, "segment source")
        self.src = src
        self.ld = src.shape[-1] if ld is None else ld
        self.C = (self.ld - c_off) if C_ is None else C_
        self.c_off, self.dy, self.dx, self.dt = c_off, dy, dx, dt


def conv_taps(srcs: Sequence[torch.Tensor], pad_lo: int = 1, ksize: int = 3) -> List[SegSpec]:
    """Segments of a kxk conv over the channel-concat of `srcs`: tap-major, source-minor -- the K order of
    weight.permute(0, 2, 3, 1) of a conv whose input channels are [srcs[0] | srcs[1] | ...]."""
    segs = []
    for ky in range(ksize):
        for kx in range(ksize):
            for s in srcs:
                segs.append(SegSpec(s, dy=ky - pad_lo, dx=kx - pad_lo))
    return segs


def temporal_taps(src: torch.Tensor) -> List[SegSpec]:
    return [SegSpec(src, dt=d) for d in (-1, 0, 1)]


class Gemm:
    """out[M, N(/2)] = epilogue(A_gather[M, K] @ W[N, K]^T): one pre-baked hi3d_gemm_params block."""

    def __init__(self, segs: Sequence[SegSpec], W: torch.Tensor, out: torch.Tensor, M: int, *, mode: int = ROWS_PLAIN,
                 geom: Optional[dict] = None, bias: Optional[torch.Tensor] = None,
                 rowbias: Optional[torch.Tensor] = None, rb_div: int = 1, rb_mod: int = 1, act: int = ACT_NONE,
                 residual: Optional[torch.Tensor] = None, blend_x: Optional[torch.Tensor] = None, alpha: float = 0.0,
                 engine: str = "mma", gn_stats: Optional[torch.Tensor] = None, gn_unit: int = 0, gn_rows: int = 0,
                 gn_partials: Optional[torch.Tensor] = None):
        _chk16(W, "W")
        _chk16(out, "out")
        Nn, K = W.shape
        if len(segs) > N.MAX_SEGS:
            raise ValueError(f"too many segments ({len(segs)})")
        p = N.GemmParams()
        p.M, p.N, p.K, p.mode = M, Nn, K, mode
        g = geom or {}
        p.Ho, p.Wo = g.get("Ho", 1), g.get("Wo", 1)
        p.Hs, p.Ws = g.get("Hs", p.Ho), g.get("Ws", p.Wo)
        p.stride, p.ups, p.T = g.get("stride", 1), g.get("ups", 0), g.get("T", 1)
        p.out_up, p.out_py, p.out_px = g.get("out_up", 0), g.get("out_py", 0), g.get("out_px", 0)
        p.Tin, p.t_off = g.get("Tin", 0), g.get("t_off", 0)
        p.nseg = len(segs)
        for i, s in enumerate(segs):
            p.seg[i].src, p.seg[i].ld, p.seg[i].c_off, p.seg[i].C = s.src.data_ptr(), s.ld, s.c_off, s.C
            p.seg[i].dy, p.seg[i].dx, p.seg[i].dt = s.dy, s.dx, s.dt
        p.W = W.data_ptr()
        if bias is not None:
            _chk32(bias, "bias")
            if bias.numel() != Nn:
                raise ValueError("bias size")
        p.bias = _ptr(bias)
        if rowbias is not None:     # may be a column slice of a wider matrix (rows of stride rb_ld)
            if rowbias.dtype != F16 or not rowbias.is_cuda or rowbias.dim() != 2 or rowbias.stride(1) != 1 \
                    or rowbias.shape[1] < Nn:
                raise ValueError("rowbias: expected CUDA fp16 [R, >=N] with unit column stride")
            p.rb_ld = rowbias.stride(0)
        p.rowbias, p.rb_div, p.rb_mod = _ptr(rowbias), rb_div, rb_mod
        p.act = act
        n_out = Nn // 2 if act == ACT_GEGLU else Nn
        if residual is not None:
            _chk16(residual, "residual")
            p.res_ld = residual.shape[-1]
        p.residual = _ptr(residual)
        if blend_x is not None:
            _chk16(blend_x, "blend_x")
            p.blend_ld = blend_x.shape[-1]
        p.blend_x, p.alpha = _ptr(blend_x), float(alpha)
        p.out, p.out_ld = out.data_ptr(), out.shape[-1]
        if out.shape[-1] < n_out or out.numel() < M * out.shape[-1] * (4 if p.out_up else 1):
            raise ValueError(f"out too small: {tuple(out.shape)} for M={M} N_out={n_out}")
        if gn_stats is not None:      # GroupNorm statistics of the output from the epilogue (hi3d_gemm_params::gn_stats)
            _chk32(gn_stats, "gn_stats")
            if gn_unit <= 0 or Nn % gn_unit or gn_rows <= 0 or M % gn_rows or gn_stats.numel() < (M // gn_rows) * (Nn // gn_unit) * 2:
                raise ValueError(f"gn_stats: unit {gn_unit} / rows {gn_rows} do not fit N={Nn}, M={M}, table {tuple(gn_stats.shape)}")
            p.gn_stats, p.gn_unit, p.gn_rows = gn_stats.data_ptr(), gn_unit, gn_rows
        self.p = p
        self._keep = (list(segs), W, out, bias, rowbias, residual, blend_x, gn_stats, gn_partials)   # keep storages alive
        self._det = ()
        if gn_stats is not None and gn_partials is not None:
            # deterministic statistics (hi3d_gemm_det / hi3d_gemm_tc5_det): gn_stats is overwritten, gn_partials is scratch
            _chk32(gn_partials, "gn_partials")
            self._det = (gn_partials.data_ptr(), gn_partials.numel())
            self._fn = N.load().hi3d_gemm_tc5_det if engine == "tc5" else N.load().hi3d_gemm_det
        else:
            self._fn = N.load().hi3d_gemm_tc5 if engine == "tc5" else N.load().hi3d_gemm
        self.flops = 2.0 * M * Nn * K
        self.out = out

    def __call__(self):
        rc = self._fn(C.byref(self.p), *self._det, _stream())
        if rc:
            N.check(rc, "hi3d_gemm")


# ------------------------------------------------------------------------------------------------------
def groupnorm_ws(n_samples: int, device) -> torch.Tensor:
    return torch.empty(int(N.load().hi3d_groupnorm_ws_floats(n_samples)), dtype=torch.float32, device=device)


def groupnorm_silu(x1: torch.Tensor, x2: Optional[torch.Tensor], n_samples: int, rows_per_sample: int,
                   gamma: torch.Tensor, beta: torch.Tensor, eps: float, silu: bool, y: torch.Tensor,
                   ws: torch.Tensor, det: bool = False):
    _chk16(x1, "x1"); _chk16(y, "y"); _chk32(gamma, "gamma"); _chk32(beta, "beta")
    c2 = 0
    if x2 is not None:
        _chk16(x2, "x2")
        c2 = x2.shape[-1]
    fn = N.load().hi3d_groupnorm_silu_det if det else N.load().hi3d_groupnorm_silu
    N.check(fn(x1.data_ptr(), x1.shape[-1], _ptr(x2), c2, n_samples, rows_per_sample,
                                         gamma.data_ptr(), beta.data_ptr(), eps, int(silu), y.data_ptr(),
                                         ws.data_ptr(), _stream()), "hi3d_groupnorm_silu")


def groupnorm_sums(x1: torch.Tensor, x2: Optional[torch.Tensor], n_samples: int, rows_per_sample: int, sums: torch.Tensor,
                   ws: torch.Tensor, det: bool = False):
    """Local (sum, sumsq) per (sample, group) -> sums fp32 [n_samples, 32, 2] (all-reduced by the caller when sharded)."""
    _chk16(x1, "x1"); _chk32(sums, "sums")
    c2 = 0 if x2 is None else x2.shape[-1]
    fn = N.load().hi3d_groupnorm_sums_det if det else N.load().hi3d_groupnorm_sums
    N.check(fn(x1.data_ptr(), x1.shape[-1], _ptr(x2), c2, n_samples, rows_per_sample,
                                         sums.data_ptr(), ws.data_ptr(), _stream()), "hi3d_groupnorm_sums")


def groupnorm_apply(x1: torch.Tensor, x2: Optional[torch.Tensor], n_samples: int, rows_per_sample: int, sums: torch.Tensor,
                    count_rows: int, gamma: torch.Tensor, beta: torch.Tensor, eps: float, silu: bool, y: torch.Tensor,
                    y_sample_rows: int = 0, y_row_off: int = 0, y_prev: Optional[int] = None, y_next: Optional[int] = None,
                    frame_rows: int = 0):
    """y_prev / y_next: raw device pointers of the SAME haloed buffer on the ranks holding the previous / next frames
    (peer memory); the boundary frames are then also stored into their halo slots (hi3d_groupnorm_apply_halo)."""
    _chk16(x1, "x1"); _chk16(y, "y"); _chk32(sums, "sums"); _chk32(gamma, "gamma"); _chk32(beta, "beta")
    c2 = 0 if x2 is None else x2.shape[-1]
    N.check(N.load().hi3d_groupnorm_apply_halo(x1.data_ptr(), x1.shape[-1], _ptr(x2), c2, n_samples, rows_per_sample,
                                               sums.data_ptr(), count_rows, gamma.data_ptr(), beta.data_ptr(), eps, int(silu),
                                               y.data_ptr(), y_sample_rows, y_row_off, y_prev, y_next, frame_rows, _stream()),
            "hi3d_groupnorm_apply")


def groupnorm_apply_stats(x1: torch.Tensor, stats1: torch.Tensor, x2: Optional[torch.Tensor], stats2: Optional[torch.Tensor],
                          unit: int, n_samples: int, rows_per_sample: int, imgs_per_sample: int, count_rows: int,
                          gamma: torch.Tensor, beta: torch.Tensor, eps: float, silu: bool, y: torch.Tensor,
                          y_sample_rows: int = 0, y_row_off: int = 0, y_prev: Optional[int] = None, y_next: Optional[int] = None,
                          frame_rows: int = 0):
    """GroupNorm(32)[+SiLU] in ONE launch: statistics from the unit tables written by the producing GEMM epilogues."""
    _chk16(x1, "x1"); _chk16(y, "y"); _chk32(stats1, "stats1"); _chk32(gamma, "gamma"); _chk32(beta, "beta")
    c2 = 0 if x2 is None else x2.shape[-1]
    if x2 is not None:
        _chk16(x2, "x2"); _chk32(stats2, "stats2")
    N.check(N.load().hi3d_groupnorm_apply_stats(x1.data_ptr(), x1.shape[-1], stats1.data_ptr(), _ptr(x2), c2, _ptr(stats2), unit,
                                                n_samples, rows_per_sample, imgs_per_sample, count_rows, gamma.data_ptr(),
                                                beta.data_ptr(), eps, int(silu), y.data_ptr(), y_sample_rows, y_row_off, y_prev,
                                                y_next, frame_rows, _stream()), "hi3d_groupnorm_apply_stats")


def groupnorm_unit_stats(x: torch.Tensor, n_images: int, rows_per_image: int, unit: int, stats: torch.Tensor,
                         partials: Optional[torch.Tensor] = None):
    """Unit table of x, accumulated into `stats`; with `partials` (scratch) deterministic, and `stats` is overwritten."""
    _chk16(x, "x"); _chk32(stats, "stats")
    if partials is not None:
        _chk32(partials, "partials")
        N.check(N.load().hi3d_groupnorm_unit_stats_det(x.data_ptr(), x.shape[-1], n_images, rows_per_image, unit, stats.data_ptr(),
                                                       partials.data_ptr(), partials.numel(), _stream()),
                "hi3d_groupnorm_unit_stats_det")
        return
    N.check(N.load().hi3d_groupnorm_unit_stats(x.data_ptr(), x.shape[-1], n_images, rows_per_image, unit, stats.data_ptr(),
                                               _stream()), "hi3d_groupnorm_unit_stats")


def groupnorm_group_sums(stats1: torch.Tensor, C1: int, stats2: Optional[torch.Tensor], C2: int, unit: int, n_samples: int,
                         imgs_per_sample: int, sums: torch.Tensor, det: bool = False):
    _chk32(stats1, "stats1"); _chk32(sums, "sums")
    fn = N.load().hi3d_groupnorm_group_sums_det if det else N.load().hi3d_groupnorm_group_sums
    N.check(fn(stats1.data_ptr(), C1, _ptr(stats2), C2, unit, n_samples, imgs_per_sample,
                                               sums.data_ptr(), _stream()), "hi3d_groupnorm_group_sums")


def groupnorm_partials_floats(n_images: int, rows_per_image: int, C: int, unit: int) -> int:
    """Scratch floats a deterministic producer of an [n_images, C / unit, 2] statistics table needs."""
    return int(N.load().hi3d_groupnorm_partials_floats(n_images, rows_per_image, C, unit))


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, y: torch.Tensor, M: int,
              addvec: Optional[torch.Tensor] = None, add_div: int = 1, add_mod: int = 1, eps: float = 1e-5):
    _chk16(x, "x"); _chk16(y, "y"); _chk32(gamma, "gamma"); _chk32(beta, "beta")
    if addvec is not None:
        _chk16(addvec, "addvec")
    N.check(N.load().hi3d_layernorm(x.data_ptr(), _ptr(addvec), add_div, add_mod, M, x.shape[-1], gamma.data_ptr(),
                                    beta.data_ptr(), eps, y.data_ptr(), _stream()), "hi3d_layernorm")


def attention_d64(qkv: torch.Tensor, n_img: int, L: int, heads: int, out: torch.Tensor, scale: float = 0.125,
                  engine: str = "mma"):
    _chk16(qkv, "qkv"); _chk16(out, "out")
    fn = N.load().hi3d_attention_d64_tc5 if engine == "tc5" else N.load().hi3d_attention_d64
    N.check(fn(qkv.data_ptr(), n_img, L, heads, scale, out.data_ptr(), _stream()), "hi3d_attention_d64")


def attention_d512(qkv: torch.Tensor, n_img: int, L: int, out: torch.Tensor, scale: float = 512 ** -0.5):
    """VAE AttnBlock core: one head of dimension 512, qkv fp16 [n_img*L, 1536] -> out fp16 [n_img*L, 512]."""
    _chk16(qkv, "qkv"); _chk16(out, "out")
    if qkv.shape[-1] != 1536 or out.shape[-1] != 512:
        raise ValueError("attention_d512: qkv must be [rows, 1536], out [rows, 512]")
    N.check(N.load().hi3d_attention_d512_tc5(qkv.data_ptr(), n_img, L, scale, out.data_ptr(), _stream()), "hi3d_attention_d512_tc5")


def temporal_attention_d64(qkv: torch.Tensor, B: int, T: int, S: int, heads: int, out: torch.Tensor,
                           scale: float = 0.125):
    _chk16(qkv, "qkv"); _chk16(out, "out")
    N.check(N.load().hi3d_temporal_attention_d64(qkv.data_ptr(), B, T, S, heads, scale, out.data_ptr(), _stream()),
            "hi3d_temporal_attention_d64")


def temporal_attention_d64_sharded(qkv_sb, out_sb, rank: int, world: int, B: int, T_local: int, S: int, heads: int,
                                   scale: float = 0.125):
    """qkv_sb / out_sb: peer.SymmBuffer of the q|k|v and output token matrices (same layout on every rank)."""
    N.check(N.load().hi3d_temporal_attention_d64_sharded(qkv_sb.ptr_array, out_sb.ptr_array, rank, world, B, T_local, S, heads,
                                                         scale, _stream()), "hi3d_temporal_attention_d64_sharded")


def softmax_rows(s: torch.Tensor, rows: int, L: int, scale: float):
    _chk16(s, "s")
    N.check(N.load().hi3d_softmax_rows(s.data_ptr(), rows, L, scale, _stream()), "hi3d_softmax_rows")


def transpose(x: torch.Tensor, R: int, Cc: int, in_ld: int, out: torch.Tensor):
    N.check(N.load().hi3d_transpose(x.data_ptr(), R, Cc, in_ld, out.data_ptr(), _stream()), "hi3d_transpose")


def timestep_embedding(t: torch.Tensor, dim: int, out: torch.Tensor, max_period: float = 10000.0):
    _chk32(t, "t"); _chk16(out, "out")
    N.check(N.load().hi3d_timestep_embedding(t.data_ptr(), t.numel(), dim, max_period, out.data_ptr(), _stream()),
            "hi3d_timestep_embedding")


def sampler_pre(x: torch.Tensor, sigma: torch.Tensor, concat_uc: Optional[torch.Tensor], concat_c: Optional[torch.Tensor],
                out: torch.Tensor, c_noise_out: Optional[torch.Tensor] = None):
    _chk32(x, "x"); _chk32(sigma, "sigma"); _chk16(out, "out")
    F_, Cx, H, W = x.shape
    Cc, is32 = 0, 0
    if concat_c is not None:
        Cc = concat_c.shape[1]
        is32 = int(concat_c.dtype == torch.float32)
        for t in (concat_c, concat_uc):
            if t is not None and (not t.is_contiguous() or t.dtype != concat_c.dtype or tuple(t.shape) != (F_, Cc, H, W)):
                raise ValueError("concat tensors must be contiguous NCHW of identical dtype/shape [F, Cc, H, W]")
    N.check(N.load().hi3d_sampler_pre(x.data_ptr(), sigma.data_ptr(), _ptr(concat_uc), _ptr(concat_c), is32, F_, Cx, Cc,
                                      H, W, out.shape[-1], out.data_ptr(), _ptr(c_noise_out), _stream()),
            "hi3d_sampler_pre")


def sampler_post(net: torch.Tensor, x: torch.Tensor, sigma: torch.Tensor, sigma_next: torch.Tensor,
                 scale: torch.Tensor, x_out: torch.Tensor, denoised_out: Optional[torch.Tensor] = None):
    _chk16(net, "net"); _chk32(x, "x"); _chk32(sigma, "sigma"); _chk32(sigma_next, "sigma_next"); _chk32(scale, "scale")
    F_, Cx, H, W = x.shape
    N.check(N.load().hi3d_sampler_post(net.data_ptr(), net.shape[-1], x.data_ptr(), sigma.data_ptr(),
                                       sigma_next.data_ptr(), scale.data_ptr(), scale.numel(), F_, Cx, H, W,
                                       x_out.data_ptr(), _ptr(denoised_out), _stream()), "hi3d_sampler_post")


def sampler_lincomb(out: torch.Tensor, terms):
    """out = sum_k c_k[f] * x_k; terms = [(x_k fp32 [F, ...], c_k fp32 [F]), ...] (1..4 terms)."""
    if not 1 <= len(terms) <= 4:
        raise ValueError("1..4 terms")
    _chk32(out, "out")
    F_ = out.shape[0]
    xs, cs = [], []
    for x, c in terms:
        _chk32(x, "x"); _chk32(c, "c")
        if x.shape != out.shape or c.numel() != F_:
            raise ValueError("lincomb: shape mismatch")
        xs.append(x.data_ptr()); cs.append(c.data_ptr())
    xs += [None] * (4 - len(xs)); cs += [None] * (4 - len(cs))
    N.check(N.load().hi3d_sampler_lincomb4(out.data_ptr(), *xs, *cs, F_, out.numel() // F_, _stream()), "hi3d_sampler_lincomb4")
    return out


def renoise_blend(lat: torch.Tensor, init: torch.Tensor, z: torch.Tensor, alpha: float, sigma: float):
    _chk32(lat, "lat"); _chk32(init, "init"); _chk32(z, "z")
    N.check(N.load().hi3d_renoise_blend(lat.data_ptr(), init.data_ptr(), z.data_ptr(), alpha, sigma, lat.numel(),
                                        _stream()), "hi3d_renoise_blend")


def nchw_to_nhwc(x: torch.Tensor, out: torch.Tensor, scale: float = 1.0):
    if not x.is_contiguous() or x.dtype not in (torch.float32, F16):
        raise ValueError("nchw_to_nhwc: contiguous fp32/fp16 NCHW expected")
    n, c, h, w = x.shape
    _chk16(out, "out")
    N.check(N.load().hi3d_nchw_to_nhwc(x.data_ptr(), int(x.dtype == torch.float32), n, c, h, w, out.shape[-1], scale,
                                       out.data_ptr(), _stream()), "hi3d_nchw_to_nhwc")


def nhwc_to_nchw(x: torch.Tensor, out: torch.Tensor, scale: float = 1.0):
    _chk16(x, "x")
    n, c, h, w = out.shape
    N.check(N.load().hi3d_nhwc_to_nchw(x.data_ptr(), x.shape[-1], n, c, h, w, scale, out.data_ptr(),
                                       int(out.dtype == torch.float32), _stream()), "hi3d_nhwc_to_nchw")


def gaussian_sample(moments: torch.Tensor, noise: Optional[torch.Tensor], out: torch.Tensor, scale: float):
    _chk16(moments, "moments"); _chk32(out, "out")
    n, c, h, w = out.shape
    if noise is not None:
        _chk32(noise, "noise")
    N.check(N.load().hi3d_gaussian_sample(moments.data_ptr(), moments.shape[-1], _ptr(noise), n, c, h, w, scale,
                                          out.data_ptr(), _stream()), "hi3d_gaussian_sample")


def pack_weight_native(w: torch.Tensor, taps: int, cin_pad: Optional[int] = None, cout_pad: Optional[int] = None,
                       geglu: bool = False) -> torch.Tensor:
    """hi3d_pack_weight (the C-ABI twin of pack.py): w = contiguous (Co, Ci, taps...) fp32 / fp16 on the device."""
    assert w.is_cuda and w.is_contiguous() and w.dtype in (torch.float32, torch.float16)
    co, ci = w.shape[0], w.shape[1]
    assert w.numel() == co * ci * taps
    cip, cop = cin_pad or ci, cout_pad or co
    out = torch.empty(cop, taps * cip, dtype=torch.float16, device=w.device)
    N.check(N.load().hi3d_pack_weight(w.data_ptr(), int(w.dtype == torch.float32), co, ci, taps, cip, cop, int(geglu),
                                      out.data_ptr(), _stream()), "hi3d_pack_weight")
    return out


def pack_bias_native(b: Optional[torch.Tensor], n: int, n_pad: Optional[int] = None, geglu: bool = False,
                     device=None) -> torch.Tensor:
    dev = b.device if b is not None else device
    out = torch.empty(n_pad or n, dtype=torch.float32, device=dev)
    is32 = int(b is None or b.dtype == torch.float32)
    N.check(N.load().hi3d_pack_bias(_ptr(b), is32, n, n_pad or n, int(geglu), out.data_ptr(), _stream()), "hi3d_pack_bias")
    return out
