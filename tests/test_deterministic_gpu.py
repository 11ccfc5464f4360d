"""Deterministic mode on the B200: every GroupNorm statistics producer gives bit-identical tables run after run (and
within fp32 rounding of an fp64 sum of the stored tensor), and with HI3D_DETERMINISTIC=1 the UNet, the samplers and the
VAE decoders give bit-identical outputs for the same weights and inputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from hi3d_official_b200 import _native, configs, ops, pack, spec  # noqa: E402
from hi3d_official_b200.unet import VideoUNet  # noqa: E402
from oracle import hi3d_oracle as O  # noqa: E402

DEV = "cuda"


def _rnd(*shape, scale=1.0, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _unit_ref(y, n_img, unit):
    """fp64 (sum, sumsq) per (image, unit) of the stored fp16 tensor y [n_img * rows, C], and the sums of |terms|."""
    v = y.double().view(n_img, -1, y.shape[-1] // unit, unit)
    return torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], -1), torch.stack([v.abs().sum((1, 3)), (v * v).sum((1, 3))], -1)


def _check_table(tabs, ref, what):
    ref, mag = ref
    for t in tabs[1:]:
        assert torch.equal(t, tabs[0]), f"{what}: statistics differ between runs"
    # fp32 rounding of the per-thread running sums (up to a few thousand terms each) relative to the sum of |terms|
    err = float(((tabs[0].double() - ref).abs() / (mag + 1.0)).max())
    print(f"[det] {what}: max err vs fp64 / sum|terms| {err:.2e}")
    assert err < 1e-4, what


def _run3(fn, stats):
    out = []
    for _ in range(3):
        stats.fill_(float("nan"))          # the deterministic producers overwrite the table: no zeroing needed
        fn()
        torch.cuda.synchronize()
        out.append(stats.clone())
    return out


def _part(n_img, rows, C, unit):
    return torch.empty(ops.groupnorm_partials_floats(n_img, rows, C, unit), dtype=torch.float32, device=DEV)


# unit sizes 4 / 10 / 20 / 40 (model_channels 128 / 320 / 640 / 1280), an 8 x 8 level (two images per 128-row tile), a
# concat consumer (two source tensors), the stage-2 level-0 shape (320 channels, 128 x 128, 32 images), a unit-2 model
@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("n,h,cin,cout,unit", [(4, 16, 64, 128, 4), (4, 16, 128, 320, 10), (2, 16, 64, 640, 20),
                                               (2, 16, 64, 1280, 40), (8, 8, 128, 320, 10), (2, 16, 64, 64, 2),
                                               (32, 128, 320, 320, 10)])
def test_tc5_conv_epilogue_statistics(n, h, cin, cout, unit, pair):
    lib = _native.load()
    lib.hi3d_gemm_tc5_set_pair_mode(pair)
    try:
        x = _rnd(n * h * h, cin, seed=1).half()
        x2 = _rnd(n * h * h, 64, seed=4).half()                  # concat: K segments from two tensors
        W = _rnd(cout, 9 * (cin + 64), scale=0.05, seed=2).half()
        b = _rnd(cout, scale=0.1, seed=3)
        out = torch.empty(n * h * h, cout, dtype=torch.float16, device=DEV)
        stats = torch.empty(n, cout // unit, 2, dtype=torch.float32, device=DEV)
        g = ops.Gemm(ops.conv_taps([x, x2]), W, out, n * h * h, mode=ops.ROWS_CONV2D, geom=dict(Ho=h, Wo=h, Hs=h, Ws=h),
                     bias=b, residual=x if cin == cout else None, engine="tc5", gn_stats=stats, gn_unit=unit, gn_rows=h * h,
                     gn_partials=_part(n, h * h, cout, unit))
        tabs = _run3(g, stats)
        _check_table(tabs, _unit_ref(out, n, unit), f"tc5 conv n={n} h={h} C={cout} unit={unit} pair={pair}")
    finally:
        lib.hi3d_gemm_tc5_set_pair_mode(-1)


@pytest.mark.parametrize("engine", ["tc5", "mma"])
def test_upconv_four_launches(engine):
    n, h, C, unit = 4, 16, 320, 10
    x = _rnd(n * h * h, C, seed=1).half()
    parity = pack.pack_upconv_parity(_rnd(C, C, 3, 3, scale=0.03, seed=2))
    out = torch.empty(n * 4 * h * h, C, dtype=torch.float16, device=DEV)
    stats = torch.empty(n, C // unit, 2, dtype=torch.float32, device=DEV)
    part = _part(n, 4 * h * h, C, unit)
    gs = [ops.Gemm([ops.SegSpec(x, dy=sy, dx=sx) for sy, sx in shifts], Wt, out, n * h * h, mode=ops.ROWS_CONV2D,
                   geom=dict(Ho=h, Wo=h, Hs=h, Ws=h, out_up=1, out_py=py, out_px=px), engine=engine, gn_stats=stats,
                   gn_unit=unit, gn_rows=h * h, gn_partials=part) for (py, px), (Wt, shifts) in parity.items()]
    tabs = _run3(lambda: [g() for g in gs], stats)
    _check_table(tabs, _unit_ref(out, n, unit), f"up-conv {engine}")


def test_temporal_and_plain_rows():
    B, T, HW, C, unit = 2, 8, 64, 320, 10
    x = _rnd(B * T * HW, C, seed=1).half()
    W = _rnd(C, 3 * C, scale=0.03, seed=2).half()
    out = torch.empty(B * T * HW, C, dtype=torch.float16, device=DEV)
    stats = torch.empty(B * T, C // unit, 2, dtype=torch.float32, device=DEV)
    g = ops.Gemm(ops.temporal_taps(x), W, out, B * T * HW, mode=ops.ROWS_TEMPORAL, geom=dict(Ho=HW, Wo=1, T=T), engine="tc5",
                 gn_stats=stats, gn_unit=unit, gn_rows=HW, gn_partials=_part(B * T, HW, C, unit))
    _check_table(_run3(g, stats), _unit_ref(out, B * T, unit), "tc5 temporal")
    W2 = _rnd(C, C, scale=0.05, seed=3).half()
    g2 = ops.Gemm([ops.SegSpec(x)], W2, out, B * T * HW, engine="tc5", gn_stats=stats, gn_unit=unit, gn_rows=HW,
                  gn_partials=_part(B * T, HW, C, unit))
    _check_table(_run3(g2, stats), _unit_ref(out, B * T, unit), "tc5 plain rows")


@pytest.mark.parametrize("C,unit,n,rows", [(320, 10, 32, 128 * 128), (64, 2, 4, 1000), (1280, 40, 2, 256)])
def test_unit_stats_group_sums_and_groupnorm(C, unit, n, rows):
    x = _rnd(n * rows, C, seed=5).half()
    stats = torch.empty(n, C // unit, 2, dtype=torch.float32, device=DEV)
    part = _part(n, rows, C, unit)
    _check_table(_run3(lambda: ops.groupnorm_unit_stats(x, n, rows, unit, stats, part), stats), _unit_ref(x, n, unit),
                 f"unit stats C={C}")
    ips = 2
    sums = torch.empty(n // ips, 32, 2, dtype=torch.float32, device=DEV)
    ref_g = tuple(r.view(n // ips, ips, 32, -1, 2).sum((1, 3)) for r in _unit_ref(x, n, unit))
    _check_table(_run3(lambda: ops.groupnorm_group_sums(stats, C, None, 0, unit, n // ips, ips, sums, det=True), sums),
                 ref_g, "group sums")
    ws = ops.groupnorm_ws(n, DEV)
    gs = torch.empty(n, 32, 2, dtype=torch.float32, device=DEV)
    _check_table(_run3(lambda: ops.groupnorm_sums(x, None, n, rows, gs, ws, det=True), gs),
                 _unit_ref(x, n, C // 32), "groupnorm sums")
    gam, bet = _rnd(C, seed=6) * 0.1 + 1, _rnd(C, seed=7) * 0.1
    ys = []
    for _ in range(3):
        y = torch.empty_like(x)
        ops.groupnorm_silu(x, None, n, rows, gam, bet, 1e-5, True, y, ws, det=True)
        ys.append(y)
    assert all(torch.equal(y, ys[0]) for y in ys)


# ---------------------------------------------------------------------------------------------------------------------
KW_S1 = dict(adm_in_channels=768, num_classes="sequential", use_checkpoint=True, in_channels=8, out_channels=4,
             model_channels=320, attention_resolutions=[4, 2, 1], num_res_blocks=2, channel_mult=[1, 2, 4, 4],
             num_head_channels=64, use_linear_in_transformer=True, transformer_depth=1, context_dim=1024,
             spatial_transformer_attn_type="softmax-xformers", extra_ff_mix_layer=True, use_spatial_context=True,
             merge_strategy="learned_with_images", video_kernel_size=[3, 1, 1])


def _net(kw, engine, seed=1):
    cfg = spec.UNetConfig.from_kwargs(**kw)
    sd = spec.synth_state_dict(spec.unet_param_shapes(cfg), seed=seed)
    net = VideoUNet(**kw)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().half()
    net.set_engine(engine)
    return net, sd


def _inputs(N, hw, T, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, 8, hw, hw, generator=g).to(DEV)
    ctx = torch.randn(N // T, 1, 1024, generator=g).to(DEV)
    ctx[0] = 0
    y = torch.randn(N // T, 768, generator=g).to(DEV)
    t = torch.full((N,), 0.7, device=DEV)
    return x, ctx, y, t


@pytest.mark.parametrize("fused", ["1", "0"])
@pytest.mark.parametrize("engine", ["tc5", "mma"])
def test_unet_bit_identical(engine, fused, monkeypatch):
    monkeypatch.setenv("HI3D_DETERMINISTIC", "1")
    monkeypatch.setenv("HI3D_GN_FUSED", fused)
    kw = dict(KW_S1, model_channels=64)
    T, hw = 8, 32
    x, ctx, y, t = _inputs(2 * T, hw, T)
    net, sd = _net(kw, engine)
    outs = [net(x, timesteps=t, context=ctx, y=y, num_video_frames=T) for _ in range(3)]
    net2, _ = _net(kw, engine)
    outs.append(net2(x, timesteps=t, context=ctx, y=y, num_video_frames=T))
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    ref = O.unet_forward({k: v.cuda() for k, v in sd.items()}, x, t, ctx, y, num_video_frames=T)
    err = (outs[0].float() - ref.float()).abs()
    assert int((err > 1e-2 + 1e-3 * ref.float().abs()).sum()) == 0


def test_full_width_unet_bit_identical(monkeypatch):
    monkeypatch.setenv("HI3D_DETERMINISTIC", "1")
    net, _ = _net(KW_S1, "tc5")
    T = 16
    x, ctx, y, t = _inputs(2 * T, 64, T, seed=3)
    a = net(x, timesteps=t, context=ctx, y=y, num_video_frames=T)
    b = net(x, timesteps=t, context=ctx, y=y, num_video_frames=T)
    assert torch.equal(a, b)


def _cond(stage, h, T, seed=5):
    g = torch.Generator().manual_seed(seed)
    cc, adm = (4, 768) if stage == 1 else (13, 512)
    x = torch.randn(T, 4, h, h, generator=g).to(DEV)
    c = dict(crossattn=torch.randn(1, 1, 1024, generator=g).to(DEV), vector=torch.randn(1, adm, generator=g).to(DEV),
             concat=(torch.randn(T, cc, h, h, generator=g) * 0.18).to(DEV))
    uc = dict(crossattn=torch.zeros_like(c["crossattn"]), vector=c["vector"], concat=torch.zeros_like(c["concat"]))
    return x, c, uc


@pytest.mark.parametrize("stage", [1, 2])
def test_samplers_and_decoders_bit_identical(stage, monkeypatch):
    """Two separately built engines with the same weights and seed: torch.equal (the exact form of the engine-reload
    check, which can only bound the difference in the default mode)."""
    monkeypatch.setenv("HI3D_DETERMINISTIC", "1")
    T, h = 4, 16
    outs = []
    for _ in range(2):
        model = configs.build_engine(stage, device=DEV, unet_overrides=dict(model_channels=64), vae_overrides=dict(ch=64),
                                     num_steps=2, num_frames=T)
        spec.synth_fill_(model, seed=1, fast=False)
        x, c, uc = _cond(stage, h, T)
        if stage == 1:
            outs.append(model.sample_stage1(c, uc, x.clone(), decode=True))
        else:
            z = _rnd(T, 4, h, h, seed=9)
            outs.append(model.sample_stage2(c, uc, x.clone(), z, decode=True))
        outs.append(model.decode_first_stage(x.clone()))
        del model
    assert torch.equal(outs[0], outs[2]) and torch.equal(outs[1], outs[3])
