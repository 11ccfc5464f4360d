"""Pins the oracle restatement (oracle/hi3d_oracle.py) and the param specs (hi3d_official_b200/spec.py)
against the UNMODIFIED reference modules, through what those modules produced on the inputs below
(tests/golden/oracle_vs_reference.pt, video_decoder_ch32.pt, reference_param_shapes.json.gz; written by
`tools/make_golden.py --only-parity` where the reference tree is present)."""
import gzip
import json
import os

import pytest
import torch

from oracle import hi3d_oracle as O
from oracle import ref_import as R
from hi3d_official_b200 import spec

G = os.path.join(os.path.dirname(__file__), "golden")
SMALL = dict(model_channels=64, channel_mult=[1, 2, 4, 4], adm_in_channels=768)


def _load(name):
    return torch.load(os.path.join(G, name), weights_only=False)


def _checkerboard(t):
    """The pixels (y, x) of t[..., H, W] with y + x even, in the order tools/make_golden.py stores them."""
    return torch.cat([t[..., 0::2, 0::2].flatten(-2), t[..., 1::2, 1::2].flatten(-2)], -1)


@pytest.fixture(scope="module")
def ref_shapes():
    """{name: [[key, shape], ...]}: the reference's state-dict layouts in their own key order."""
    with gzip.open(os.path.join(G, "reference_param_shapes.json.gz"), "rt") as f:
        return json.load(f)


def _as_dict(pairs):
    return {k: tuple(s) for k, s in pairs}


@pytest.fixture(scope="module")
def fix():
    return _load("oracle_vs_reference.pt")


@pytest.fixture(scope="module")
def small_unet(ref_shapes):
    cfg = spec.UNetConfig.from_kwargs(**dict(R.UNET_S1, **SMALL))
    shapes = spec.unet_param_shapes(cfg)
    assert dict(shapes) == _as_dict(ref_shapes["unet_small"])
    return spec.synth_state_dict(shapes, seed=1)


def test_unet_param_spec_full_size_matches_reference_on_meta(ref_shapes):
    for tag, kw in (("unet_s1", R.UNET_S1), ("unet_s2", R.UNET_S2)):
        mine = spec.unet_param_shapes(spec.UNetConfig.from_kwargs(**kw))
        assert dict(mine) == _as_dict(ref_shapes[tag])
        assert sum(torch.Size(s).numel() for s in mine.values()) in (1524623082, 1524321322)


def test_unet_forward_matches_reference(small_unet, fix):
    sd = small_unet
    T = 4
    f = fix["unet_forward"]
    with torch.no_grad():
        b = O.unet_forward(sd, f["xin"], f["t"], f["ctx"], f["y"], num_video_frames=T)
    a = f["out"]
    assert a.abs().mean() > 1e-2
    torch.testing.assert_close(b, a, rtol=1e-4, atol=2e-4)


def test_sampler_matches_reference(small_unet, fix):
    sd = small_unet
    T, steps = 4, 3
    f = fix["sampler"]
    with torch.no_grad():
        b = O.sample(sd, f["x"].clone(), f["c"], f["uc"], num_steps=steps, max_scale=2.5, num_frames=T)
    torch.testing.assert_close(b, f["out"], rtol=1e-4, atol=1e-3)


def test_sampler_constants(fix):
    s = O.edm_sigmas(25)
    torch.testing.assert_close(s, fix["edm_sigmas_25"], rtol=0, atol=0)
    assert abs(float(s[0]) - 700.0001) < 1e-3 and float(s[-1]) == 0.0 and abs(float(s[-2]) - 0.002) < 1e-6
    cs = O.vscaling_edm_cnoise(torch.tensor(700.0))
    assert abs(float(cs[3]) - 1.6377701) < 1e-6 and abs(float(cs[2]) - 1.4285699e-03) < 1e-9
    assert abs(O.v02_alpha(1) - 0.984126) < 1e-6 and O.v02_alpha(0) == 1.0


def test_single_key_cross_attention_is_constant(small_unet):
    """SURVEY F7: attn2 with one context token == to_out(to_v(ctx)) for every query."""
    sd = small_unet
    pre = "input_blocks.1.1.transformer_blocks.0.attn2."
    x = torch.randn(3, 10, 64)
    ctx = torch.randn(3, 1, 1024)
    full = O.cross_attention(sd, pre, x, ctx, 1)
    const = torch.nn.functional.linear(torch.nn.functional.linear(ctx, sd[pre + "to_v.weight"]),
                                       sd[pre + "to_out.0.weight"], sd[pre + "to_out.0.bias"])
    torch.testing.assert_close(full, const.expand_as(full), rtol=1e-5, atol=1e-6)


def test_vae_matches_reference(ref_shapes, fix):
    cfg = spec.VAEConfig.from_ddconfig(dict(R.VAE_DD, ch=32), 4)
    shapes = spec.vae_param_shapes(cfg)
    assert dict(shapes) == _as_dict(ref_shapes["vae_ch32"])
    sd = spec.synth_state_dict(shapes, seed=2)
    f = fix["vae"]
    img = f["img"]
    with torch.no_grad():
        torch.testing.assert_close(O.vae_encode(sd, img, scale_factor=1.0), f["z_mode"], rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(O.vae_decode(sd, f["z"], scale_factor=1.0), f["dec"], rtol=1e-4, atol=2e-4)
        # sampled posterior: the reference draws CPU randn (distributions.py:37-41); `noise` is that draw
        torch.testing.assert_close(O.vae_encode(sd, img, noise=f["noise"], scale_factor=1.0), f["z_sampled"], rtol=1e-4, atol=1e-4)


def test_vae_full_size_spec_on_meta(ref_shapes):
    mine = {k: v for k, v in spec.vae_param_shapes(spec.VAEConfig.from_ddconfig(R.VAE_DD, 4)).items()
            if not k.startswith(("quant_conv", "post_quant_conv"))}
    assert mine == _as_dict(ref_shapes["vae_encoder_decoder"])


@pytest.mark.parametrize("vks", [[3, 1, 1], 3])
def test_video_decoder_oracle_matches_reference(vks, ref_shapes):
    """SURVEY §8(f) N1: the oracle restatement of temporal_ae.VideoDecoder (time_mode 'conv-only'; kernel (3,1,1) as in
    SVD and the full 3x3x3 default) against the unmodified reference class, seeded synthetic weights drawn in the
    reference's state-dict order; the reference's output is stored as its checkerboard half."""
    f = _load("video_decoder_ch32.pt")[f"vks{vks}"]
    g = torch.Generator().manual_seed(11)
    sd = {}
    for k, shape in ref_shapes[f"video_decoder_ch32_vks{vks}"]:
        if k.endswith("mix_factor"):
            sd[k] = torch.full(shape, 0.3)
        elif len(shape) == 1 and ("norm" in k or "in_layers.0" in k or "out_layers.0" in k) and k.endswith("weight"):
            sd[k] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif len(shape) == 1:
            sd[k] = 0.05 * torch.randn(shape, generator=g)
        else:                       # incl. the zero_module'd out_layers conv of every time_stack (F8)
            fan_in = torch.Size(shape[1:]).numel()
            sd[k] = torch.randn(shape, generator=g) * fan_in ** -0.5
    T = 3
    z = torch.randn(2 * T, 4, 8, 8, generator=g)
    assert torch.equal(z, f["z"])           # the same draws as the reference run
    with torch.no_grad():
        b = O.vae_video_decoder({"decoder." + k: v for k, v in sd.items()}, z, T)
        b2 = O.vae_video_decoder({"decoder." + k: v for k, v in sd.items()}, z.flip(0), T).flip(0)
    assert b.shape == (2 * T, 3, 64, 64)
    torch.testing.assert_close(_checkerboard(b), f["out_checkerboard"], rtol=1e-4, atol=2e-4)
    torch.testing.assert_close(_checkerboard(b2), f["flipped_checkerboard"], rtol=1e-4, atol=2e-4)
    # the temporal branch matters: shuffling the frames changes more than a permutation of the output
    assert (f["flipped_checkerboard"] - f["out_checkerboard"]).abs().max() > 1e-3


@pytest.mark.parametrize("vks", [[3, 1, 1], 3])
def test_video_decoder_param_spec_matches_reference_on_meta(vks, ref_shapes):
    mine = spec.video_decoder_param_shapes(spec.VAEConfig.from_ddconfig(R.VAE_DD, 4), vks)
    assert dict(mine) == _as_dict(ref_shapes[f"video_decoder_vks{vks}"])
