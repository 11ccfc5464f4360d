"""CPU-side tests: the C-ABI library loads and exports every declared symbol, block topology / param specs,
weight packing, the generic (reference-API) sampler path against the oracle, config glue, loud failure on CPU."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from hi3d_official_b200 import _native, configs, pack, sampling, spec, util
from oracle import hi3d_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = _native.load()
    hdr = open(os.path.join(ROOT, "include", "hi3d_b200.h")).read()
    declared = set(re.findall(r"\b(hi3d_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    for s in declared:
        assert hasattr(lib, s)
    assert lib.hi3d_abi_version() == 2
    # parameter-block layout must match the C struct: 17 ints (+4 pad), 24 segs of 32 bytes, then the tail
    assert _native.GemmParams.seg.offset == 72 and _native.Seg.__dict__["dt"].offset == 28
    import ctypes
    assert ctypes.sizeof(_native.Seg) == 32


def test_unet_topology_matches_survey_census():
    cfg = spec.UNetConfig.from_kwargs(**configs.UNET_STAGE1)
    plan = spec.unet_plan(cfg)
    layers = [L for b in plan.input_blocks + [plan.middle] + plan.output_blocks for L in b]
    assert len(plan.input_blocks) == 12 and len(plan.output_blocks) == 12
    assert sum(L.kind == "res" for L in layers) == 22 and sum(L.kind == "attn" for L in layers) == 16
    assert [L.cin for L in layers if L.kind == "res" and L.name.startswith("output_blocks")] == \
        [2560, 2560, 2560, 2560, 2560, 1920, 1920, 1280, 960, 960, 640, 640]
    shapes = spec.unet_param_shapes(cfg)
    assert len(shapes) == 1428
    assert sum(torch.Size(s).numel() for s in shapes.values()) == 1524623082
    cfg2 = spec.UNetConfig.from_kwargs(**configs.UNET_STAGE2)
    assert sum(torch.Size(s).numel() for s in spec.unet_param_shapes(cfg2).values()) == 1524321322
    v = spec.vae_param_shapes(spec.VAEConfig.from_ddconfig(configs._VAE_DD, 4))
    assert len(v) == 248 and abs(sum(torch.Size(s).numel() for s in v.values()) - 83.65e6) < 0.05e6


def test_unsupported_variants_fail_loudly():
    with pytest.raises(NotImplementedError):
        spec.UNetConfig.from_kwargs(**dict(configs.UNET_STAGE1, use_scale_shift_norm=True))
    with pytest.raises(NotImplementedError):
        spec.UNetConfig.from_kwargs(**dict(configs.UNET_STAGE1, video_kernel_size=[3, 3, 3]))
    with pytest.raises(NotImplementedError):
        spec.VAEConfig.from_ddconfig(dict(configs._VAE_DD, attn_resolutions=[32]))


def test_conv_packing_matches_tap_order():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 6, 5, 7, generator=g)
    w = torch.randn(4, 6, 3, 3, generator=g)
    ref = F.conv2d(x, w, padding=1)
    Wp = pack.pack_conv2d(w).float()                       # [Co, 9*Ci], (ky, kx, ci)
    xp = F.pad(x, (1, 1, 1, 1)).permute(0, 2, 3, 1)        # NHWC
    cols = torch.cat([xp[:, ky:ky + 5, kx:kx + 7] for ky in range(3) for kx in range(3)], -1)
    out = (cols.half().float() @ Wp.t()).permute(0, 3, 1, 2)
    torch.testing.assert_close(out, ref, rtol=2e-2, atol=2e-2)
    # padded variants keep the real block and zero the rest
    Wpad = pack.pack_conv2d(w, cin_pad=64, cout_pad=8).view(8, 3, 3, 64)
    assert torch.equal(Wpad[:4, :, :, :6], w.permute(0, 2, 3, 1).half()) and float(Wpad[4:].abs().sum()) == 0
    # temporal conv: (kt, ci)
    wt = torch.randn(4, 6, 3, 1, 1, generator=g)
    assert torch.equal(pack.pack_conv3d_t(wt).view(4, 3, 6), wt[:, :, :, 0, 0].permute(0, 2, 1).half())
    # GEGLU interleave
    wg, bg = torch.randn(16, 5, generator=g), torch.randn(16, generator=g)
    wi, bi = pack.pack_geglu(wg, bg)
    assert torch.equal(wi[0::2], wg[:8].half()) and torch.equal(wi[1::2], wg[8:].half())
    assert torch.equal(bi[0::2], bg[:8]) and torch.equal(bi[1::2], bg[8:])


def test_generic_sampler_path_matches_oracle_with_a_toy_network():
    """EulerEDMSampler / Denoiser / LinearPredictionGuider generic path (any callable denoiser), on CPU."""
    T = 4
    lin = torch.nn.Conv2d(8, 4, 1)

    class Net(torch.nn.Module):
        def forward(self, x, t, c, **kw):
            return lin(torch.cat([x, c["concat"]], 1)) * t.view(-1, 1, 1, 1).cos()
    net = Net()
    den = sampling.Denoiser({"target": "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise"})
    smp = sampling.EulerEDMSampler(
        num_steps=5, device="cpu",
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization", "params": {"sigma_max": 700.0}},
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
                       "params": {"num_frames": T, "max_scale": 2.5, "min_scale": 1.0}})
    g = torch.Generator().manual_seed(1)
    x = torch.randn(T, 4, 6, 6, generator=g)
    c = dict(crossattn=torch.randn(1, 1, 8, generator=g), vector=torch.randn(1, 8, generator=g),
             concat=torch.randn(T, 4, 6, 6, generator=g))
    uc = dict(crossattn=torch.zeros(1, 1, 8), vector=c["vector"], concat=torch.zeros(T, 4, 6, 6))
    with torch.no_grad():
        out = smp(lambda i, s, cc: den(net, i, s, cc), x.clone(), cond=c, uc=uc)
        # oracle loop with the same toy network
        sig = O.edm_sigmas(5)
        torch.testing.assert_close(smp.discretization(5), sig, rtol=0, atol=0)
        xr = x * torch.sqrt(1.0 + sig[0] ** 2.0)
        scale = O.guider_scale(T, 2.5)
        for i in range(5):
            s = torch.full((2 * T,), float(sig[i]))
            c_skip, c_out, c_in, c_noise = O.vscaling_edm_cnoise(s.view(-1, 1, 1, 1))
            xin = torch.cat([xr, xr])
            d = net(xin * c_in, c_noise.view(-1), {"concat": torch.cat([uc["concat"], c["concat"]])}) * c_out + xin * c_skip
            du, dc = d.chunk(2)
            dd = du + scale.view(-1, 1, 1, 1) * (dc - du)
            xr = xr + (xr - dd) / sig[i] * (sig[i + 1] - sig[i])
    torch.testing.assert_close(out, xr, rtol=1e-5, atol=1e-4)
    # step_call == one iteration of __call__
    x0 = x * torch.sqrt(1.0 + sig[0] ** 2.0)
    with torch.no_grad():
        a = smp.step_call(lambda i, s, cc: den(net, i, s, cc), x0, 0, x0.new_ones(T), sig, len(sig), c, uc)
        b = smp.sampler_step(x0.new_ones(T) * sig[0], x0.new_ones(T) * sig[1], lambda i, s, cc: den(net, i, s, cc), x0, c, uc)
    torch.testing.assert_close(a, b)


def test_known_answer_constants():
    """SURVEY App. C."""
    s = sampling.EDMDiscretization(sigma_max=700.0)(25)
    assert s.shape == (26,) and abs(float(s[1]) - 545.7295) < 1e-2 and abs(float(s[12]) - 15.58997) < 1e-3
    sc = sampling.VScalingWithEDMcNoise()(torch.tensor(0.002))
    assert abs(float(sc[0]) - 0.99999595) < 1e-6 and abs(float(sc[3]) + 1.5536520) < 1e-5
    gdr = sampling.LinearPredictionGuider(2.0, 16)
    assert torch.allclose(gdr.scale[0], torch.linspace(1, 2, 16))


def test_config_glue_resolves_reference_targets_and_builds_on_meta():
    assert util.get_obj_from_str("sgm.modules.diffusionmodules.video_model.VideoUNet").__module__ == "hi3d_official_b200.unet"
    cfg = configs.stage1_config()["model"]
    cfg["params"]["network_config"]["params"]["model_channels"] = 64
    cfg["params"]["first_stage_config"]["params"]["ddconfig"]["ch"] = 64
    m = util.get_obj_from_str(cfg["target"])(**cfg["params"])
    keys = set(m.state_dict())
    assert "model.diffusion_model.input_blocks.1.1.time_stack.0.attn1.to_q.weight" in keys
    assert "first_stage_model.decoder.up.3.upsample.conv.weight" in keys and "first_stage_model.quant_conv.weight" in keys
    assert m.num_samples == 16 and m.scale_factor == 0.18215 and m.sampler.num_steps == 25
    assert isinstance(m.sampler.guider, sampling.LinearPredictionGuider) and m.sampler.guider.max_scale == 2.5
    with pytest.raises(RuntimeError, match="no CPU fallback"):          # product path refuses to compute off-GPU
        m.model.diffusion_model(torch.zeros(8, 8, 8, 8), timesteps=torch.zeros(8), context=torch.zeros(2, 1, 1024),
                                y=torch.zeros(2, 768), num_video_frames=4)
    c = {"crossattn": torch.ones(1, 1, 1024), "vector": torch.ones(1, 768), "concat": torch.ones(16, 4, 8, 8)}
    cc, uc = m.conditioner.get_unconditional_conditioning({"c": c}, force_uc_zero_embeddings=["cond_frames"])
    assert float(uc["crossattn"].abs().sum()) == 0 and float(uc["concat"].abs().sum()) == 0 and torch.equal(uc["vector"], c["vector"])


@pytest.mark.parametrize("name,adm,cin", [("inference-v01.yaml", 768, 8), ("inference-v02.yaml", 512, 17)])
def test_unmodified_reference_yaml_instantiates(name, adm, cin):
    """The reference's inference configs, stored parsed (JSON is YAML) under tests/golden/ by tools/make_golden.py."""
    from hi3d_official_b200 import engine
    with torch.device("meta"):
        m = engine.create_model(os.path.join(ROOT, "tests", "golden", name.replace(".yaml", ".json")))
    u = m.model.diffusion_model
    assert u.cfg.adm_in_channels == adm and u.in_channels == cin and m.en_and_decode_n_samples_a_time in (1, 16)
    assert type(m).__name__ in ("VideoLDM", "VideoLDMStage2")


def test_checkpoint_loader_accepts_reference_layouts(tmp_path):
    cfg = configs.stage1_config()["model"]
    cfg["params"]["network_config"]["params"]["model_channels"] = 64
    cfg["params"]["first_stage_config"]["params"]["ddconfig"]["ch"] = 64
    m = util.get_obj_from_str(cfg["target"])(**cfg["params"])
    spec.synth_fill_(m, seed=3)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    ds = tmp_path / "first_stage.pt"                        # DeepSpeed layout: {'module': {'module.<k>': v}}
    torch.save({"module": {"module." + k: v for k, v in sd.items()}}, ds)
    ck = tmp_path / "x.ckpt"
    torch.save({"state_dict": dict(sd, **{"conditioner.embedders.0.foo": torch.zeros(1)})}, ck)
    for path in (ds, ck):
        m2 = util.get_obj_from_str(cfg["target"])(**cfg["params"])
        m2.init_from_ckpt(str(path))
        for k, v in m2.state_dict().items():
            assert torch.equal(v, sd[k]), k


def test_flop_count_matches_survey():
    """tools/count_flops.py (plan-derived) against the reference-graph figures of SURVEY.md §8(d)."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sp = importlib.util.spec_from_file_location("count_flops", os.path.join(root, "tools", "count_flops.py"))
    cf = importlib.util.module_from_spec(sp)
    sp.loader.exec_module(cf)
    for stage, survey in ((1, 4.061e13), (2, 2.095e14)):
        per, ref, ours = cf.count(stage)
        assert abs(ref - survey) / survey < 0.01, (stage, ref, survey)
        assert 0.90 * ref < ours < ref          # the folds remove a few per cent, nothing else


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm): exactly one stdout line with the keys every bench line carries."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--ref-latent", "8", "--ref-budget-s", "120"], capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    # the unmodified reference modules wherever they can be imported (the reference tree, or the copy oracle/build_ref.py
    # staged under oracle/_ref); without them the arm times the oracle port and says so
    from oracle import ref_import as R
    assert d["impl"] == "reference" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == ("reference" if R.available() else "port")
    assert d["config"]["reference_latent_override"] == 8 and d["sampler_steps_timed"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_video_io_and_svd_widening(tmp_path):
    """SURVEY 8f N3: tensor2vid / export_to_video (vtdm/util.py:12-49) and the 8 -> 17 channel / 768 -> 512 checkpoint surgery
    (tool_make_init_svd_to_vid2vid.py:40-61) against their definitions."""
    import numpy as np
    from hi3d_official_b200 import configs, spec, video_io
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, 16), torch.linspace(-1, 1, 24), indexing="ij")
    v = torch.stack([torch.stack([xx * (0.5 + 0.1 * f), yy, -xx * yy]) for f in range(4)], 1)[None]   # smooth (codec-friendly)
    v = v + torch.tensor([1.3, -1.3, 0.0]).view(1, 3, 1, 1, 1) * 0.2                                 # some values clamp
    ref = ((v.clone() * 0.5 + 0.5).clamp(0, 1).permute(0, 2, 3, 4, 1).reshape(4, 16, 24, 3).numpy() * 255).astype("uint8")
    frames = video_io.tensor2vid(v.clone())
    assert len(frames) == 4 and frames[0].shape == (16, 24, 3) and frames[0].dtype == np.uint8
    assert all(np.array_equal(a, b) for a, b in zip(frames, ref))
    mp4 = video_io.export_to_video(frames, str(tmp_path / "first.mp4"), fps=8)
    back = video_io.read_video_frames(mp4)
    assert len(back) == 4 and back[0].shape == (16, 24, 3)
    assert np.abs(back[0].astype(int) - frames[0].astype(int)).mean() < 12          # lossy codec: same picture, not same bits
    gif = video_io.export_to_video(frames, str(tmp_path / "first.mp4"), save_to_gif=True)
    assert gif.endswith(".gif") and (tmp_path / "first.gif").exists()
    # checkpoint surgery on reduced-width configs (same rule at every width)
    kw1, kw2 = dict(configs.UNET_STAGE1, model_channels=32), dict(configs.UNET_STAGE2, model_channels=32)
    sd1 = spec.synth_state_dict(spec.unet_param_shapes(spec.UNetConfig.from_kwargs(**kw1)), seed=3)
    sd2 = spec.synth_state_dict(spec.unet_param_shapes(spec.UNetConfig.from_kwargs(**kw2)), seed=4)
    pre = "model.diffusion_model."
    wide = video_io.widen_svd_state_dict({pre + k: t for k, t in sd1.items()}, {pre + k: t for k, t in sd2.items()})
    w_in, w1 = wide[pre + "input_blocks.0.0.weight"], sd1["input_blocks.0.0.weight"]
    assert w_in.shape[1] == 17 and torch.equal(w_in[:, :4], w1[:, :4]) and torch.equal(w_in[:, 13:], w1[:, 4:])
    assert not bool(w_in[:, 4:13].any())
    le, l1 = wide[pre + "label_emb.0.0.weight"], sd1["label_emb.0.0.weight"]
    assert le.shape[1] == 512 and not bool(le[:, :256].any()) and torch.equal(le[:, 256:], l1[:, 512:])
    same = [k for k in sd1 if k not in ("input_blocks.0.0.weight", "label_emb.0.0.weight")]
    assert all(torch.equal(wide[pre + k], sd1[k]) for k in same)


def test_docs_point_at_existing_profiles():
    """Every `profiles/r0N_*` file the documents cite exists (brace lists and globs expanded)."""
    import glob
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def expand(name):
        m = re.search(r"\{([^}]*)\}", name)
        if not m:
            return [name]
        out = []
        for alt in m.group(1).split(","):
            out += expand(name[:m.start()] + alt + name[m.end():])
        return out

    missing = []
    for doc in ("DESIGN.md", "README.md", "profiles/README.md", "INTEGRATION.md"):
        text = open(os.path.join(root, doc)).read()
        for m in re.finditer(r"`((?:profiles/)?r0[12]_[A-Za-z0-9_{},.*-]+)`", text):
            ref = m.group(1) if m.group(1).startswith("profiles/") else "profiles/" + m.group(1)
            for f in expand(ref):
                if not glob.glob(os.path.join(root, f)) and not glob.glob(os.path.join(root, f) + "*"):
                    missing.append((doc, f))
    assert not missing, missing
