"""SURVEY §8f N2: the conditioner pieces that need no third-party weights, against the unmodified reference classes
(their outputs and the reference's inference-v02 config, stored under tests/golden/ by `tools/make_golden.py
--only-parity`) and against their definitions."""
import os

import pytest
import torch

from hi3d_official_b200 import conditioner as Cn
from hi3d_official_b200 import util

G = os.path.join(os.path.dirname(__file__), "golden")


def _golden():
    return torch.load(os.path.join(G, "conditioner.pt"), weights_only=False)


def test_concat_timestep_embedder_matches_reference():
    for x, ref in _golden()["timestep_embedder"]:
        torch.testing.assert_close(Cn.ConcatTimestepEmbedderND(256)(x), ref, rtol=1e-5, atol=1e-5)


def test_video_prediction_embedder_arrangement_matches_reference():
    """Frame / copy bookkeeping of VideoPredictionEmbedderWithEncoder (modules.py:1012-1021) with an identity 'encoder'."""
    cfg = {"target": "torch.nn.Identity"}
    fix = _golden()["video_prediction"]
    vid = torch.arange(2 * 3 * 4 * 5 * 5, dtype=torch.float32).reshape(6, 4, 5, 5)      # (b t) = 2 x 3 cond frames
    assert torch.equal(vid, fix["vid"])
    for ncf, ncp in ((3, 1), (1, 4), (3, 2)):
        mine = Cn.VideoPredictionEmbedderWithEncoder(ncf, ncp, cfg, scale_factor=0.5)
        torch.testing.assert_close(mine(vid.clone()), fix["out"][(ncf, ncp)])


def test_depth_pixel_unshuffle_and_normalisation():
    """vtdm/encoders.py:44-50: channel k = h0 * 3 + w0 of output pixel (i, j) is the normalised depth at (3 i + h0, 3 j + w0)."""
    g = torch.Generator().manual_seed(1)
    y = torch.rand(2, 20, 28, generator=g) * 7 + 3
    out = Cn.depth_to_concat(y, 64, 96, shuffle_size=3)
    assert out.shape == (2, 9, 8, 12)
    up = torch.nn.functional.interpolate(y[:, None], [24, 36], mode="bilinear")
    for i in range(2):
        up[i] -= up[i].min()
        up[i] /= max(float(up[i].max()), 1e-6)
    from einops import rearrange
    torch.testing.assert_close(out, rearrange(up, "b c (h h0) (w w0) -> b (c h0 w0) h w", h0=3, w0=3))
    assert float(out.min()) == 0.0 and abs(float(out.amax(dim=(1, 2, 3)).min()) - 1.0) < 1e-6


def test_clip_embedder_bookkeeping_and_aes_vector():
    e = Cn.FrozenOpenCLIPImagePredictionEmbedder({"target": "sgm.modules.encoders.modules.FrozenOpenCLIPImageEmbedder",
                                                  "params": {"version": "x", "freeze": True}}, n_cond_frames=1, n_copies=1)
    with pytest.raises(NotImplementedError, match="third-party tower"):
        e(torch.zeros(1, 3, 8, 8))
    e.open_clip.set_fn(lambda v: torch.ones(v.shape[0], 1024) * v.mean())
    assert e(torch.full((2, 3, 8, 8), 0.5)).shape == (2, 1, 1024)
    a = Cn.AesEmbedder()
    a.scorer.set_fn(lambda y: torch.full((y.shape[0], 1), 5.5))
    x = torch.rand(2, 3, 16, 64, 64) * 2 - 1
    v = a(x)
    assert v.shape == (2, 256) and float(v[0, 0]) == 5.5
    torch.testing.assert_close(v[:, 1:], Cn.timestep_embedding(torch.tensor([550.0, 550.0]), 255))
    assert a.preprocess(x).shape == (2, 3, 224, 224)


def test_unmodified_conditioner_config_produces_reference_shaped_conditioning():
    """The conditioner_config of the UNMODIFIED inference-v02.yaml (stored parsed, as JSON), with the towers' outputs
    supplied in the batch and a stub in place of the VAE encoder: keys, shapes, concat order [depth 9 | latent 4],
    vector = [elevation | cond_aug], and the force_uc_zero_embeddings semantics of pipeline_i2v_eval_v02.py:111-118."""
    cfg = util.load_yaml(os.path.join(G, "inference-v02.json"))["model"]["params"]["conditioner_config"]
    with torch.device("meta"):
        cond = util.instantiate_from_config(cfg)
    names = [type(e).__name__ for e in cond.embedders]
    assert names == ["FrozenOpenCLIPImagePredictionEmbedder", "ConcatTimestepEmbedderND", "DepthEmbedder",
                     "VideoPredictionEmbedderWithEncoder", "ConcatTimestepEmbedderND"]

    class FakeAE(torch.nn.Module):
        def encode(self, x):
            return torch.nn.functional.avg_pool2d(x, 8)[:, [0, 1, 2, 0]] * 2.0
    cond.embedders[3].encoder = FakeAE()
    T, H = 16, 64
    g = torch.Generator().manual_seed(2)
    frames = torch.rand(T, 3, H, H, generator=g) * 2 - 1
    batch = {"cond_frames_without_noise": frames[:1], "cond_frames_without_noise:clip": torch.randn(1, 1024, generator=g),
             "elevation": torch.tensor([10.0]), "cond_aug": torch.tensor([0.02]), "cond_frames": frames,
             "cond_frames:depth": torch.rand(T, 24, 24, generator=g)}
    c, uc = cond.get_unconditional_conditioning(batch, force_uc_zero_embeddings=["cond_frames", "cond_frames_without_noise"])
    assert c["crossattn"].shape == (1, 1, 1024) and c["vector"].shape == (1, 512) and c["concat"].shape == (T, 13, 8, 8)
    torch.testing.assert_close(c["concat"][:, :9], Cn.depth_to_concat(batch["cond_frames:depth"], H, H, 3))
    torch.testing.assert_close(c["concat"][:, 9:], FakeAE().encode(frames))
    torch.testing.assert_close(c["vector"][:, :256], Cn.timestep_embedding(torch.tensor([10.0]), 256))
    assert not bool(uc["crossattn"].any()) and not bool(uc["concat"].any()) and torch.equal(uc["vector"], c["vector"])
