#!/usr/bin/env python
"""Stage-1 entry point, same CLI as the reference's pipeline_i2v_eval_v01.py (:39-45) on the B200 engine.

    python pipeline_i2v_eval_v01.py --denoise_config configs/inference-v01.yaml --denoise_checkpoint ckpts/first_stage.pt \
        --image_path demo/15_out.png --output_dir outputs/15_out --elevation 0  [--cond cond.pt | --synthetic]

The hot path (25-step fused Euler-EDM over VideoUNet + VAE decode) runs here.  The third-party conditioner towers (rembg,
OpenCLIP ViT-H, CLIP-L + aesthetic MLP) are outside it; three ways to supply what they produce:
  --towers t.pt   {'clip': (1, 1024) image embedding, 'aes': (1, 1) aesthetic score}: the image is pre-processed as in the
                  reference (cv2 resize, centre crop, [-1, 1]; v01:131-149), `add_custom_cond` and the model's own
                  GeneralConditioner (elevation / cond_aug timestep embeddings, VAE-mode latent of the cond frame) build c / uc
                  exactly like v01:62-78;
  --cond c.pt     torch.save({'c': .., 'uc': ..}) from the reference's conditioner.get_unconditional_conditioning;
  --synthetic     seeded stand-ins.
Output: <output_dir>/first_step/first.mp4 (8 fps, like v01:96-98,129) + first.pt (the frames as a tensor, which stage 2
prefers over re-reading the lossy mp4).  Without a checkpoint file the seeded synthetic weights of spec.synth_fill_ are used
(said loudly).  --tiny builds a reduced-width 2-step model: the smoke size the tests execute this script at.
"""
import argparse
import os
import random

import torch

from hi3d_official_b200 import configs, spec
from hi3d_official_b200.engine import create_model
from hi3d_official_b200.util import get_obj_from_str


def load_model(config_path, ckpt, stage, tiny=False):
    if os.path.exists(config_path) and not tiny:
        model = create_model(config_path)
    else:
        if not tiny:
            print(f"[hi3d-b200] {config_path} not found: using the built-in copy of the stage-{stage} inference config")
        cfg = (configs.stage1_config(True) if stage == 1 else configs.stage2_config(True))["model"]
        if tiny:
            cfg["params"]["network_config"]["params"]["model_channels"] = 64
            cfg["params"]["first_stage_config"]["params"]["ddconfig"]["ch"] = 64
            cfg["params"]["sampler_config"]["params"]["num_steps"] = 2
            for e in cfg["params"]["conditioner_config"]["params"]["emb_models"]:
                if "encoder_config" in e.get("params", {}):
                    e["params"]["encoder_config"]["params"]["ddconfig"]["ch"] = 64
        model = get_obj_from_str(cfg["target"])(**cfg["params"])
    if os.path.exists(ckpt):
        model.init_from_ckpt(ckpt)
        model = model.cuda().half()
    else:
        print(f"[hi3d-b200] checkpoint {ckpt} not found: SEEDED SYNTHETIC WEIGHTS (outputs are not images)")
        model = model.cuda().half()
        spec.synth_fill_(model, seed=0, fast=True)
    return model


def synthetic_cond(stage, T, h, device, seed):
    g = torch.Generator().manual_seed(seed)
    adm, cc = (768, 4) if stage == 1 else (512, 13)
    c = dict(crossattn=torch.randn(1, 1, 1024, generator=g), vector=torch.randn(1, adm, generator=g),
             concat=(torch.randn(T, cc, h, h, generator=g) * 0.18).half())
    c = {k: v.to(device) for k, v in c.items()}
    uc = dict(crossattn=torch.zeros_like(c["crossattn"]), vector=c["vector"].clone(), concat=torch.zeros_like(c["concat"]))
    return c, uc


def save_frames(frames, out_dir, name, fps=8):
    """frames: (T, 3, H, W) in [-1, 1] -> <out_dir>/<name>.mp4 through tensor2vid / export_to_video (vtdm/util.py:12-49,
    v01:96-98) and <out_dir>/<name>.pt."""
    from hi3d_official_b200 import video_io
    os.makedirs(out_dir, exist_ok=True)
    torch.save(frames.cpu(), os.path.join(out_dir, name + ".pt"))
    vid = frames.float().cpu().permute(1, 0, 2, 3)[None]                      # "t c h w -> 1 c t h w"
    return video_io.export_to_video(video_io.tensor2vid(vid.clone()), os.path.join(out_dir, name + ".mp4"), fps=fps)


def load_image(path, size):
    """v01:131-149: cv2 read -> resize so the short side is `size` -> centre crop -> [-1, 1], (3, size, size)."""
    import cv2
    import numpy as np
    img = cv2.cvtColor(cv2.imread(path), cv2.COLOR_BGR2RGB)
    hh, ww = img.shape[:2]
    sc = size / min(hh, ww)
    img = cv2.resize(img, (max(size, round(ww * sc)), max(size, round(hh * sc))), interpolation=cv2.INTER_AREA)
    y0, x0 = (img.shape[0] - size) // 2, (img.shape[1] - size) // 2
    img = img[y0:y0 + size, x0:x0 + size]
    return torch.from_numpy(np.ascontiguousarray(img)).permute(2, 0, 1).float() / 127.5 - 1.0


def cond_from_towers(model, frames, towers, elevation, stage):
    """v01:62-78 / v02:104-118: batch -> add_custom_cond -> GeneralConditioner with the third-party towers' outputs supplied.
    frames: (3, T, H, W) in [-1, 1] on the GPU (stage 1: the image repeated T times)."""
    T = model.num_samples
    batch = {"video": frames[None], "elevation": torch.tensor([float(elevation)], device=frames.device),
             "fps_id": torch.tensor([7.0], device=frames.device), "motion_bucket_id": torch.tensor([127.0], device=frames.device)}
    batch = model.add_custom_cond(batch, infer=True)
    batch["cond_frames_without_noise:clip"] = towers["clip"].to(frames.device).float().reshape(1, -1)
    if stage == 1:
        batch["video:aes"] = towers["aes"].to(frames.device).float().reshape(1, 1)
    else:
        batch["cond_frames:depth"] = towers["depth"].to(frames.device).float()
    c, uc = model.conditioner.get_unconditional_conditioning(
        batch, force_uc_zero_embeddings=["cond_frames", "cond_frames_without_noise"])
    return c, uc


def enable_deterministic():
    """--deterministic: the same seed and inputs give bit-identical frames (same GPU type, build and configuration).  Set
    before CUDA is initialised, so that cuBLAS in the torch-side conditioner is covered too; the engine's launch plans
    then use the deterministic GroupNorm statistics (hi3d_official_b200.ops.deterministic)."""
    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    torch.use_deterministic_algorithms(True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--denoise_config", type=str, default="configs/inference-v01.yaml")
    ap.add_argument("--denoise_checkpoint", type=str, default="ckpts/first_stage.pt")
    ap.add_argument("--image_path", type=str, default="demo/15_out.png")
    ap.add_argument("--output_dir", type=str, default="outputs/15_out")
    ap.add_argument("--elevation", type=int, default=0)
    ap.add_argument("--cond", type=str, default=None)
    ap.add_argument("--towers", type=str, default=None)
    ap.add_argument("--synthetic", action="store_true")
    ap.add_argument("--tiny", action="store_true")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--deterministic", action="store_true", help="bit-identical output for the same seed and inputs")
    params = ap.parse_args()
    if params.deterministic:
        enable_deterministic()
    seed = random.randint(0, 65535) if params.seed is None else params.seed      # v01:33-34
    torch.manual_seed(seed)
    model = load_model(params.denoise_config, params.denoise_checkpoint, 1, params.tiny)
    T = model.num_samples                                                        # 16 frames
    h = 16 if params.tiny else 64                                                # 512^2 / 8
    if params.cond:
        d = torch.load(params.cond, map_location="cuda")
        c, uc = d["c"], d["uc"]
    elif params.towers:
        img = load_image(params.image_path, 8 * h).cuda()
        c, uc = cond_from_towers(model, img[:, None].repeat(1, T, 1, 1), torch.load(params.towers), params.elevation, 1)
    elif params.synthetic:
        c, uc = synthetic_cond(1, T, h, "cuda", seed)
    else:
        raise SystemExit("the conditioner towers are outside the B200 hot path: pass --towers / --cond <file> or --synthetic")
    randn = torch.randn(T, 4, h, h, device="cuda")                               # v01:91
    with torch.no_grad():
        frames = model.sample_stage1(c, uc, randn)                               # v01:92-94
    mp4 = save_frames(frames, os.path.join(params.output_dir, "first_step"), "first")
    print(f"[hi3d-b200] wrote {T} frames {tuple(frames.shape[1:])} to {mp4} (seed {seed})")


if __name__ == "__main__":
    main()
