"""Parity against fixtures produced by the UNMODIFIED reference (tools/make_golden.py, CPU fp32):
  * not-gpu: the oracle restatement reproduces them (pins the oracle where /root/reference is absent);
  * gpu: the CUDA path meets the north-star tolerance on the CFG-combined denoised latents D(x, sigma)
    (teacher-forced: rtol 1e-3, atol 1e-2, fp16) and on the VAE encode / decode."""
import os

import pytest
import torch

from oracle import hi3d_oracle as O
from hi3d_official_b200 import spec

G = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return torch.load(os.path.join(G, name), weights_only=False)


def _checkerboard(t):
    """The pixels (y, x) of t[..., H, W] with y + x even, in the order tools/make_golden.py stores them."""
    return torch.cat([t[..., 0::2, 0::2].flatten(-2), t[..., 1::2, 1::2].flatten(-2)], -1)


def _unet_sd(fix):
    return spec.synth_state_dict(spec.unet_param_shapes(spec.UNetConfig.from_kwargs(**fix["unet_kwargs"])), seed=fix["seed"])


@pytest.mark.parametrize("tag", ["s1", "s2"])
def test_oracle_reproduces_reference_unet_fixture(tag):
    fix = _load(f"unet_{tag}_mc64.pt")
    sd = _unet_sd(fix)
    T = fix["T"]
    scale = O.guider_scale(T, fix["max_scale"])
    with torch.no_grad():
        for sigma, ref in fix["denoised"].items():
            xs = fix["x"] * (1 + sigma ** 2) ** 0.5
            d = O.cfg_denoise(sd, xs, torch.full((T,), sigma), fix["c"], fix["uc"], scale, num_video_frames=T)
            torch.testing.assert_close(d, ref, rtol=1e-4, atol=2e-4)
            e = O.euler_step(sd, xs, sigma, sigma * 0.7, fix["c"], fix["uc"], scale, num_video_frames=T)
            torch.testing.assert_close(e, fix["euler"][sigma], rtol=1e-4, atol=2e-3)
        s3 = O.sample(sd, fix["x"].clone(), fix["c"], fix["uc"], num_steps=3, max_scale=fix["max_scale"], num_frames=T)
        torch.testing.assert_close(s3, fix["sampled3"], rtol=1e-4, atol=1e-3)


def test_oracle_reproduces_reference_vae_fixture():
    fix = _load("vae_ch64.pt")
    sd = spec.synth_state_dict(spec.vae_param_shapes(spec.VAEConfig.from_ddconfig(fix["ddconfig"], 4)), seed=fix["seed"])
    with torch.no_grad():
        torch.testing.assert_close(O.vae_encode(sd, fix["img"], scale_factor=1.0), fix["z_mode"], rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(O.vae_encode(sd, fix["img"], noise=fix["noise"], scale_factor=1.0), fix["z_sampled"],
                                   rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(O.vae_decode(sd, fix["z_in"], scale_factor=1.0), fix["dec"], rtol=1e-4, atol=2e-4)


def test_oracle_reproduces_reference_video_decoder_fixture():
    """SURVEY 8f N1: fixture from the unmodified temporal_ae.VideoDecoder (tools/make_golden.py --only-video); its output
    is stored as the checkerboard half of the pixels."""
    fix = _load("vae_video_ch64.pt")
    cfg = spec.VAEConfig.from_ddconfig(fix["ddconfig"], 4)
    sd = spec.synth_state_dict(spec.video_decoder_param_shapes(cfg, tuple(fix["video_kernel_size"])), seed=fix["seed"])
    with torch.no_grad():
        torch.testing.assert_close(_checkerboard(O.vae_video_decoder(sd, fix["z"], fix["T"])), fix["dec_checkerboard"],
                                   rtol=1e-4, atol=2e-4)


# ------------------------------------------------------------------------------------------------------------------
def _stats(a, b, name, rtol=1e-3, atol=1e-2):
    err = (a.float() - b.float()).abs()
    frac = float((err > atol + rtol * b.abs()).float().mean())
    print(f"[{name}] max|err| {float(err.max()):.3e} mean|err| {float(err.mean()):.3e} ref mean|x| "
          f"{float(b.abs().mean()):.3e} frac outside {frac:.2e}")
    return float(err.max()), frac


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["s1", "s2"])
def test_cuda_unet_meets_north_star_tolerance_on_reference_fixture(tag):
    from hi3d_official_b200 import sampling
    from hi3d_official_b200.unet import VideoUNet
    fix = _load(f"unet_{tag}_mc64.pt")
    net = VideoUNet(**fix["unet_kwargs"])
    net.load_state_dict(_unet_sd(fix), strict=True)
    net = net.cuda().half()
    T = fix["T"]
    dev = "cuda"
    c = {k: v.to(dev) for k, v in fix["c"].items()}
    uc = {k: v.to(dev) for k, v in fix["uc"].items()}
    den = sampling.Denoiser({"target": "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise"})
    fd = sampling.FusedDenoiser(den, sampling.OpenAIWrapper(net), num_video_frames=T,
                                image_only_indicator=torch.zeros(2, T, device=dev))
    smp = sampling.EulerEDMSampler(
        num_steps=3, device=dev,
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization", "params": {"sigma_max": 700.0}},
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
                       "params": {"num_frames": T, "max_scale": fix["max_scale"], "min_scale": 1.0}})
    for sigma, ref in fix["denoised"].items():
        xs = (fix["x"] * (1 + sigma ** 2) ** 0.5).to(dev)
        s = torch.full((T,), sigma, device=dev)
        # fused path (product): sampler_pre -> plan -> sampler_post, returns the guided denoised latents too
        st = smp._fused_state(fd, xs, c, uc, refresh=True)
        assert st is not None, "fused path not taken"
        x_next, d = st.step(xs, s, s * 0.7, want_denoised=True)
        mx, frac = _stats(d.cpu(), ref, f"{tag} fused D(x,{sigma})")
        assert frac == 0.0, "north-star tolerance (rtol 1e-3, atol 1e-2) violated"
        _, frac = _stats(x_next.cpu(), fix["euler"][sigma], f"{tag} fused euler({sigma})", atol=1e-2 * max(1.0, sigma * 0.3))
        assert frac == 0.0
        # generic path (drop-in API: reference-style closure through Denoiser / OpenAIWrapper / guider)
        dg = smp.denoise(xs, lambda i, sg, cc: den(sampling.OpenAIWrapper(net), i, sg, cc, num_video_frames=T), s, c, uc)
        mx, frac = _stats(dg.cpu(), ref, f"{tag} generic D(x,{sigma})")
        assert frac == 0.0
    out = smp(fd, fix["x"].clone().to(dev), cond=c, uc=uc)
    mx, frac = _stats(out.cpu(), fix["sampled3"], f"{tag} free-running 3-step sample")
    assert frac < 1e-3


@pytest.mark.gpu
def test_cuda_vae_on_reference_fixture():
    from hi3d_official_b200.vae import AutoencoderKL, AutoencoderKLModeOnly
    fix = _load("vae_ch64.pt")
    sd = spec.synth_state_dict(spec.vae_param_shapes(spec.VAEConfig.from_ddconfig(fix["ddconfig"], 4)), seed=fix["seed"])
    ae = AutoencoderKL(embed_dim=4, ddconfig=fix["ddconfig"], lossconfig={"target": "torch.nn.Identity"}, monitor="val/rec_loss")
    ae.load_state_dict(sd, strict=True)
    ae = ae.cuda().half()
    img = fix["img"].cuda().half()
    z = ae.encode(img, noise=fix["noise"].cuda())
    mx, frac = _stats(z.cpu(), fix["z_sampled"], "vae encode (sampled)", atol=2e-2)
    assert frac == 0.0
    torch.manual_seed(77)                      # the reference's CPU-RNG draw order (distributions.py:37-41)
    z2 = ae.encode(img)
    _, frac = _stats(z2.cpu(), fix["z_sampled"], "vae encode (own CPU randn)", atol=2e-2)
    assert frac == 0.0
    mo = AutoencoderKLModeOnly(embed_dim=4, ddconfig=fix["ddconfig"])
    mo.load_state_dict(sd, strict=True)
    mo = mo.cuda().half()
    _, frac = _stats(mo.encode(img).cpu(), fix["z_mode"], "vae encode (mode)", atol=2e-2)
    assert frac == 0.0
    dec = ae.decode(fix["z_in"].cuda().half())
    mx, frac = _stats(dec.cpu(), fix["dec"], "vae decode", atol=2e-2)
    assert frac == 0.0


@pytest.mark.gpu
def test_cuda_video_decoder_on_reference_fixture():
    """SURVEY 8f N1: AutoencoderKLTemporal.decode(z, timesteps=T) -- VideoResBlocks ((3,1,1) time_stack, GroupNorm over
    (T,H,W), blend weighing the temporal branch) and the AE3DConv output conv -- against the fixture produced by the
    unmodified temporal_ae.VideoDecoder, and through DiffusionEngine.decode_first_stage's timesteps hook."""
    from hi3d_official_b200.vae import AutoencoderKLTemporal, VideoDecoder
    fix = _load("vae_video_ch64.pt")
    cfg = spec.VAEConfig.from_ddconfig(fix["ddconfig"], 4)
    sd_dec = spec.synth_state_dict(spec.video_decoder_param_shapes(cfg, (3, 1, 1)), seed=fix["seed"])
    sd_2d = spec.synth_state_dict(spec.vae_param_shapes(cfg), seed=fix["seed"])
    ae = AutoencoderKLTemporal(embed_dim=4, ddconfig=fix["ddconfig"], video_kernel_size=[3, 1, 1], time_mode="conv-only")
    sd = {k: v for k, v in sd_2d.items() if not k.startswith("decoder.")}
    sd.update(sd_dec)
    # the fixture ran the bare VideoDecoder: make post_quant_conv the identity (1x1, 4 -> 4)
    sd["post_quant_conv.weight"] = torch.eye(4).view(4, 4, 1, 1)
    sd["post_quant_conv.bias"] = torch.zeros(4)
    ae.load_state_dict(sd, strict=True)
    ae = ae.cuda().half()
    assert isinstance(ae.decoder, VideoDecoder)
    T = fix["T"]
    dec = ae.decode(fix["z"].cuda().half(), timesteps=T)
    assert dec.shape == (2 * T, 3, 128, 128)
    mx, frac = _stats(_checkerboard(dec.cpu()), fix["dec_checkerboard"], f"video decoder (T={T}, 2 clips)", atol=2e-2)
    assert frac == 0.0
    # frames matter: a frame-reversed clip is not the frame-reversed output (temporal convs / (T,H,W) statistics are live)
    dec_r = ae.decode(fix["z"].flip(0).cuda().half(), timesteps=T).flip(0)
    assert float((dec_r.float() - dec.float()).abs().max()) > 1e-2
    with pytest.raises(ValueError):
        ae.decode(fix["z"].cuda().half())                       # the temporal decoder needs timesteps
    with pytest.raises(NotImplementedError):
        AutoencoderKLTemporal(embed_dim=4, ddconfig=fix["ddconfig"], video_kernel_size=3)
