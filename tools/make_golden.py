#!/usr/bin/env python
"""Generates tests/golden/* by running the UNMODIFIED reference modules (imported read-only through
oracle/ref_import.py, which locates the reference tree) on seeded synthetic weights + inputs, CPU fp32.  The
reference is not part of this repository, so these small fixtures are what pins parity in the test suite.  Re-run
only where the reference tree is present:

    python tools/make_golden.py [--only-video | --only-parity]

Outputs larger than a fixture should be are stored as their checkerboard half (`checkerboard`), which keeps every
frame, channel, row and column.
"""
import gzip
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import as R  # noqa: E402
from hi3d_official_b200 import spec  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
UNET_KW = dict(R.UNET_S1, model_channels=64)
UNET2_KW = dict(R.UNET_S2, model_channels=64)
VAE_DD = dict(R.VAE_DD, ch=64)


def checkerboard(t):
    """The pixels (y, x) of t[..., H, W] with y + x even, as [..., H * W / 2]."""
    return torch.cat([t[..., 0::2, 0::2].flatten(-2), t[..., 1::2, 1::2].flatten(-2)], -1)


def cond(T, cc, adm, hw, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(T, 4, hw, hw, generator=g)
    c = dict(crossattn=torch.randn(1, 1, 1024, generator=g), vector=torch.randn(1, adm, generator=g),
             concat=torch.randn(T, cc, hw, hw, generator=g) * 0.18)
    uc = dict(crossattn=torch.zeros(1, 1, 1024), vector=c["vector"].clone(), concat=torch.zeros(T, cc, hw, hw))
    return x, c, uc


@torch.no_grad()
def video_decoder_fixture():
    """SURVEY 8f N1: the unmodified temporal_ae.VideoDecoder (time_mode 'conv-only', video_kernel_size [3, 1, 1]) run as
    Decoder.forward(z, timesteps=T) on seeded synthetic weights, 2 clips x 4 frames, 16x16 latents."""
    R.setup()
    from sgm.modules.autoencoding.temporal_ae import VideoDecoder
    dd = dict(VAE_DD, attn_type="vanilla")
    cfg = spec.VAEConfig.from_ddconfig(VAE_DD, 4)
    sd = spec.synth_state_dict(spec.video_decoder_param_shapes(cfg, (3, 1, 1)), seed=2)
    ref = VideoDecoder(**dd, video_kernel_size=[3, 1, 1], time_mode="conv-only").eval()
    ref.load_state_dict({k[len("decoder."):]: v for k, v in sd.items()}, strict=True)
    T = 4
    g = torch.Generator().manual_seed(8)
    z = torch.randn(2 * T, 4, 16, 16, generator=g)
    out = ref(z, timesteps=T)
    fix = dict(ddconfig=VAE_DD, seed=2, T=T, z=z, dec_checkerboard=checkerboard(out), video_kernel_size=[3, 1, 1])
    torch.save(fix, os.path.join(OUT, "vae_video_ch64.pt"))
    print("video decoder", tuple(out.shape), float(out.abs().mean()))


def _shapes(module, prefix=""):
    """[[key, shape], ...] of a state dict, in its own order."""
    return [[prefix + k, list(v.shape)] for k, v in module.state_dict().items()]


def _parity_inputs(cin_cat=4, adm=768, hw=16, T=4, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(T, 4, hw, hw, generator=g)
    c = dict(crossattn=torch.randn(1, 1, 1024, generator=g), vector=torch.randn(1, adm, generator=g),
             concat=torch.randn(T, cin_cat, hw, hw, generator=g) * 0.18)
    uc = dict(crossattn=torch.zeros(1, 1, 1024), vector=c["vector"].clone(), concat=torch.zeros(T, cin_cat, hw, hw))
    return x, c, uc


@torch.no_grad()
def parity_fixtures():
    """What tests/test_oracle_vs_reference.py, test_samplers_cpu.py, test_conditioner_cpu.py and the config tests of
    test_host_cpu.py compare with: the reference's parameter layouts, its outputs on the tests' inputs, and its two
    inference configs (parsed YAML, written as JSON)."""
    R.setup()
    from sgm.models.autoencoder import AutoencoderKL  # noqa: F401  (registers the reference's autoencoder modules)
    from sgm.modules.autoencoding.temporal_ae import VideoDecoder
    from sgm.modules.diffusionmodules.model import Decoder, Encoder
    from sgm.modules.diffusionmodules.video_model import VideoUNet
    shapes, fix = {}, {}
    # ---- parameter layouts (meta device: full size costs nothing)
    for tag, kw in (("unet_s1", R.UNET_S1), ("unet_s2", R.UNET_S2)):
        with torch.device("meta"):
            shapes[tag] = _shapes(VideoUNet(**kw))
    with torch.device("meta"):
        shapes["vae_encoder_decoder"] = _shapes(Encoder(**R.VAE_DD), "encoder.") + _shapes(Decoder(**R.VAE_DD), "decoder.")
    for vks in ([3, 1, 1], 3):
        with torch.device("meta"):
            ref = VideoDecoder(**dict(R.VAE_DD, attn_type="vanilla"), video_kernel_size=vks, time_mode="conv-only")
        shapes[f"video_decoder_vks{vks}"] = _shapes(ref, "decoder.")
    # ---- small UNet forward and 3-step sampler (weights: spec.synth_state_dict seed 1)
    small = dict(model_channels=64, channel_mult=[1, 2, 4, 4], adm_in_channels=768)
    torch.manual_seed(0)
    ref = R.build_unet(**small)
    shapes["unet_small"] = _shapes(ref)
    ref.load_state_dict(spec.synth_state_dict(spec.unet_param_shapes(spec.UNetConfig.from_kwargs(**dict(R.UNET_S1, **small))),
                                              seed=1), strict=True)
    T = 4
    x, c, uc = _parity_inputs(T=T)
    xin = torch.cat([torch.cat([x, x]), torch.cat([uc["concat"], c["concat"]])], 1)
    t = torch.full((2 * T,), 0.7)
    ctx = torch.cat([uc["crossattn"], c["crossattn"]])
    y = torch.cat([uc["vector"], c["vector"]])
    out = ref(xin, timesteps=t, context=ctx, y=y, num_video_frames=T, image_only_indicator=torch.zeros(2, T))
    fix["unet_forward"] = dict(xin=xin, t=t, ctx=ctx, y=y, out=out)
    x, c, uc = _parity_inputs(T=T, seed=3)
    smp, den, net = R.build_sampler(num_steps=3, max_scale=2.5, num_frames=T), R.build_denoiser(), R.wrap(ref)
    kw = dict(image_only_indicator=torch.zeros(2, T), num_video_frames=T)
    out = smp(lambda inp, s, cc: den(net, inp, s, cc, **kw), x.clone(), cond=c, uc=uc)
    fix["sampler"] = dict(x=x, c=c, uc=uc, out=out)
    fix["edm_sigmas_25"] = R.build_sampler().discretization(25, device="cpu")
    # ---- VAE ch=32 (weights: spec.synth_state_dict seed 2); inputs drawn after the reference's own init, so stored
    torch.manual_seed(0)
    ref = R.build_vae(sample=False, ch=32, ch_mult=[1, 2, 4, 4])
    shapes["vae_ch32"] = _shapes(ref)
    ref.load_state_dict(spec.synth_state_dict(spec.vae_param_shapes(spec.VAEConfig.from_ddconfig(dict(R.VAE_DD, ch=32), 4)),
                                              seed=2), strict=True)
    img = torch.rand(2, 3, 64, 64) * 2 - 1
    z_mode = ref.encode(img)
    z = torch.randn(2, 4, 8, 8)
    dec = ref.decode(z)
    ref.regularization.sample = True
    torch.manual_seed(7)
    z_sampled = ref.encode(img)
    torch.manual_seed(7)
    noise = torch.randn(2, 4, 8, 8)
    fix["vae"] = dict(img=img, z_mode=z_mode, z=z, dec=dec, noise=noise, z_sampled=z_sampled)
    # ---- VideoDecoder ch=32, 2 clips x 3 frames of 8x8 latents, both kernel sizes; output and frame-reversed output
    vdec = {}
    for vks in ([3, 1, 1], 3):
        torch.manual_seed(0)
        dd = dict(R.VAE_DD, ch=32, ch_mult=[1, 2, 4, 4], attn_type="vanilla")
        ref = VideoDecoder(**dd, video_kernel_size=vks, time_mode="conv-only").eval()
        shapes[f"video_decoder_ch32_vks{vks}"] = _shapes(ref)
        g = torch.Generator().manual_seed(11)
        sd = {}
        for k, v in ref.state_dict().items():
            if k.endswith("mix_factor"):
                sd[k] = torch.full_like(v, 0.3)
            elif v.ndim == 1 and ("norm" in k or "in_layers.0" in k or "out_layers.0" in k) and k.endswith("weight"):
                sd[k] = 1.0 + 0.1 * torch.randn(v.shape, generator=g)
            elif v.ndim == 1:
                sd[k] = 0.05 * torch.randn(v.shape, generator=g)
            else:
                sd[k] = torch.randn(v.shape, generator=g) * v[0].numel() ** -0.5
        ref.load_state_dict(sd, strict=True)
        T = 3
        z = torch.randn(2 * T, 4, 8, 8, generator=g)
        vdec[f"vks{vks}"] = dict(z=z, out_checkerboard=checkerboard(ref(z, timesteps=T)),
                                 flipped_checkerboard=checkerboard(ref(z.flip(0), timesteps=T).flip(0)))
    torch.save(fix, os.path.join(OUT, "oracle_vs_reference.pt"))
    torch.save(vdec, os.path.join(OUT, "video_decoder_ch32.pt"))
    with open(os.path.join(OUT, "reference_param_shapes.json.gz"), "wb") as raw, \
            gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        f.write(json.dumps(shapes, separators=(",", ":")).encode())
    print("oracle parity", {k: float(v["out"].abs().mean()) for k, v in fix.items() if isinstance(v, dict) and "out" in v})
    samplers_fixture()
    conditioner_fixture()
    for name in ("inference-v01", "inference-v02"):
        import yaml
        with open(os.path.join(R.REF_ROOT, "configs", name + ".yaml")) as f:
            cfg = yaml.safe_load(f)
        with open(os.path.join(OUT, name + ".json"), "w") as f:
            json.dump(cfg, f, indent=1)
            f.write("\n")


@torch.no_grad()
def samplers_fixture():
    """Euler / Heun / DPM-Solver++(2M) under three guiders on the analytic toy denoiser of tests/test_samplers_cpu.py."""
    import importlib.util
    R.setup()
    import sgm.modules.diffusionmodules.sampling as RS
    sp = importlib.util.spec_from_file_location("_samplers_test", os.path.join(ROOT, "tests", "test_samplers_cpu.py"))
    tm = importlib.util.module_from_spec(sp)
    sp.loader.exec_module(tm)
    T = 4
    g = torch.Generator().manual_seed(3)
    c = dict(vector=torch.randn(T, 8, generator=g), crossattn=torch.randn(T, 1, 16, generator=g),
             concat=torch.randn(T, 4, 6, 6, generator=g))
    uc = dict(vector=torch.randn(T, 8, generator=g), crossattn=torch.zeros(T, 1, 16), concat=torch.zeros(T, 4, 6, 6))
    x0 = torch.randn(4, 4, 6, 6, generator=torch.Generator().manual_seed(9))
    fix = dict(c=c, uc=uc, x0=x0, out={})
    for name in ("EulerEDMSampler", "HeunEDMSampler", "DPMPP2MSampler"):
        for guider, gcfg in tm.GUIDERS.items():
            smp = getattr(RS, name)(num_steps=7, device="cpu", verbose=False, discretization_config=tm.DISC, guider_config=gcfg)
            fix["out"][f"{name}/{guider}"] = smp(tm.toy_denoiser, x0.clone(), cond=c, uc=uc)
    torch.save(fix, os.path.join(OUT, "samplers.pt"))


@torch.no_grad()
def conditioner_fixture():
    """ConcatTimestepEmbedderND and VideoPredictionEmbedderWithEncoder (identity encoder) on the inputs of
    tests/test_conditioner_cpu.py."""
    R.setup()
    from sgm.modules.encoders.modules import ConcatTimestepEmbedderND, VideoPredictionEmbedderWithEncoder
    g = torch.Generator().manual_seed(0)
    ts = []
    for x in (torch.rand(3, generator=g) * 30, torch.rand(2, 3, generator=g) * 5, torch.tensor([0.02])):
        ts.append((x, ConcatTimestepEmbedderND(256)(x)))
    vid = torch.arange(2 * 3 * 4 * 5 * 5, dtype=torch.float32).reshape(6, 4, 5, 5)
    vp = {}
    for ncf, ncp in ((3, 1), (1, 4), (3, 2)):
        ref = VideoPredictionEmbedderWithEncoder(n_cond_frames=ncf, n_copies=ncp, encoder_config={"target": "torch.nn.Identity"},
                                                 scale_factor=0.5, disable_encoder_autocast=True)
        vp[(ncf, ncp)] = ref(vid.clone())
    torch.save(dict(timestep_embedder=ts, video_prediction=dict(vid=vid, out=vp)), os.path.join(OUT, "conditioner.pt"))


@torch.no_grad()
def main():
    os.makedirs(OUT, exist_ok=True)
    if "--only-video" in sys.argv:
        video_decoder_fixture()
        return
    if "--only-parity" in sys.argv:
        parity_fixtures()
        return
    torch.manual_seed(0)
    # ---- stage-1 style UNet (8 input channels), T=4, 16x16 latents: denoiser outputs at 3 sigmas + 3-step sampler
    for tag, kw, cc, adm, scale in (("s1", UNET_KW, 4, 768, 2.5), ("s2", UNET2_KW, 13, 512, 2.0)):
        T, hw = 4, 16
        ref = R.build_unet(**kw)
        sd = spec.synth_state_dict(spec.unet_param_shapes(spec.UNetConfig.from_kwargs(**kw)), seed=1)
        ref.load_state_dict(sd, strict=True)
        net, den = R.wrap(ref), R.build_denoiser()
        x, c, uc = cond(T, cc, adm, hw, seed=11)
        kwm = dict(image_only_indicator=torch.zeros(2, T), num_video_frames=T)
        smp = R.build_sampler(num_steps=3, max_scale=scale, num_frames=T)
        fix = dict(unet_kwargs=kw, seed=1, T=T, hw=hw, x=x, c=c, uc=uc, max_scale=scale, denoised={}, euler={})
        for sigma in (700.0, 10.0, 0.5):
            xs = x * (1 + sigma ** 2) ** 0.5
            s = torch.full((T,), sigma)
            d = smp.denoise(xs, lambda i, sg, cc_: den(net, i, sg, cc_, **kwm), s, c, uc)     # CFG-combined D(x, sigma)
            fix["denoised"][sigma] = d
            fix["euler"][sigma] = smp.sampler_step(s, s * 0.7, lambda i, sg, cc_: den(net, i, sg, cc_, **kwm), xs, c, uc)
        fix["sampled3"] = smp(lambda i, sg, cc_: den(net, i, sg, cc_, **kwm), x.clone(), cond=c, uc=uc)
        torch.save(fix, os.path.join(OUT, f"unet_{tag}_mc64.pt"))
        print(tag, {k: float(v.abs().mean()) for k, v in fix["denoised"].items()}, float(fix["sampled3"].abs().mean()))
    # ---- VAE ch=64: mode-encode, sampled encode (CPU RNG, as the reference draws it), decode
    ae = R.build_vae(sample=True, **{k: v for k, v in VAE_DD.items()})
    sdv = spec.synth_state_dict(spec.vae_param_shapes(spec.VAEConfig.from_ddconfig(VAE_DD, 4)), seed=2)
    ae.load_state_dict(sdv, strict=True)
    g = torch.Generator().manual_seed(5)
    img = torch.rand(2, 3, 128, 128, generator=g) * 2 - 1
    z_in = torch.randn(2, 4, 16, 16, generator=g)
    torch.manual_seed(77)
    z_sampled = ae.encode(img)
    torch.manual_seed(77)
    noise = torch.randn(2, 4, 16, 16)
    ae.regularization.sample = False
    fix = dict(ddconfig=VAE_DD, seed=2, img=img, z_in=z_in, noise=noise, z_mode=ae.encode(img), z_sampled=z_sampled,
               dec=ae.decode(z_in))
    torch.save(fix, os.path.join(OUT, "vae_ch64.pt"))
    print("vae", float(fix["z_mode"].abs().mean()), float(fix["dec"].abs().mean()))
    video_decoder_fixture()
    parity_fixtures()


if __name__ == "__main__":
    main()
