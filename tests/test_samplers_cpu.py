"""The sampler / guider surface of hi3d_official_b200.sampling against the UNMODIFIED reference classes
(sgm/modules/diffusionmodules/sampling.py, guiders.py) on CPU with an analytic toy denoiser: the step algebra of
Euler (fused path excluded: plain callable), Heun and DPM-Solver++(2M) (SURVEY §8(f) N4) must agree to fp32 rounding.
The reference's results are stored in tests/golden/samplers.pt (`tools/make_golden.py --only-parity`)."""
import os

import pytest
import torch

from hi3d_official_b200 import sampling as S

DISC = {"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization", "params": {"sigma_max": 700.0}}
GUIDERS = {
    "identity": None,
    "vanilla": {"target": "sgm.modules.diffusionmodules.guiders.VanillaCFG", "params": {"scale": 3.0}},
    "linear": {"target": "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
               "params": {"num_frames": 4, "max_scale": 2.5, "min_scale": 1.0}},
}


def toy_denoiser(x, sigma, c):
    """Smooth in x and sigma, depends on the conditioning: D = a x + (1 - a) tanh(mean(vector)),  a = 1 / (1 + sigma^2)."""
    a = (1.0 / (1.0 + sigma ** 2)).reshape(-1, 1, 1, 1)
    v = torch.tanh(c["vector"].mean(dim=1)).reshape(-1, 1, 1, 1)
    if v.shape[0] != x.shape[0]:
        v = v.repeat_interleave(x.shape[0] // v.shape[0], 0)
    return a * x + (1.0 - a) * v


@pytest.fixture(scope="module")
def golden():
    return torch.load(os.path.join(os.path.dirname(__file__), "golden", "samplers.pt"), weights_only=False)


@pytest.mark.parametrize("guider", list(GUIDERS))
@pytest.mark.parametrize("name", ["EulerEDMSampler", "HeunEDMSampler", "DPMPP2MSampler"])
def test_sampler_matches_reference(name, guider, golden):
    kw = dict(num_steps=7, device="cpu", verbose=False, discretization_config=DISC, guider_config=GUIDERS[guider])
    mine = getattr(S, name)(**kw)
    c, uc, x0 = golden["c"], golden["uc"], golden["x0"]
    a = golden["out"][f"{name}/{guider}"]
    with torch.no_grad():
        b = mine(toy_denoiser, x0.clone(), cond=c, uc=uc)
    assert torch.isfinite(a).all()
    assert torch.allclose(a, b, rtol=1e-5, atol=1e-5), float((a - b).abs().max())


def test_samplers_resolve_from_reference_target_strings():
    from hi3d_official_b200.util import instantiate_from_config
    for cls in ("EulerEDMSampler", "HeunEDMSampler", "DPMPP2MSampler"):
        s = instantiate_from_config({"target": f"sgm.modules.diffusionmodules.sampling.{cls}",
                                     "params": dict(num_steps=3, device="cpu", discretization_config=DISC)})
        assert type(s).__module__ == "hi3d_official_b200.sampling" and type(s).__name__ == cls
