#!/usr/bin/env python
"""Stage-2 (1024^2 refiner) entry point, same CLI as the reference's pipeline_i2v_eval_v02.py (:38-44) on the B200
engine.  Reads <output_dir>/first_step/first.pt (stage-1 frames written by pipeline_i2v_eval_v01.py; first.mp4 through
OpenCV when the tensor is absent, like v02:169-176), up-samples them to 1024^2, VAE-encodes each frame (posterior sample,
CPU RNG like the reference), runs the 25-step re-noise/blend loop of pipeline_i2v_eval_v02.py:127-135 on the fused sampler,
decodes and writes second_step_video/second.mp4.  Conditioning: --towers {'clip': (1,1024), 'depth': (T,h',w') MiDaS maps} /
--cond / --synthetic as in v01; --tiny = the smoke size the tests run."""
import argparse
import os
import random

import torch
import torch.nn.functional as F

from pipeline_i2v_eval_v01 import cond_from_towers, enable_deterministic, load_model, save_frames, synthetic_cond


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--denoise_config", type=str, default="configs/inference-v02.yaml")
    ap.add_argument("--denoise_checkpoint", type=str, default="ckpts/second_stage.pt")
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
    seed = random.randint(0, 65535) if params.seed is None else params.seed
    torch.manual_seed(seed)
    model = load_model(params.denoise_config, params.denoise_checkpoint, 2, params.tiny)
    T = model.num_samples
    h = 32 if params.tiny else 128
    first = os.path.join(params.output_dir, "first_step", "first.pt")
    first_mp4 = os.path.join(params.output_dir, "first_step", "first.mp4")
    if os.path.exists(first):
        frames = torch.load(first).cuda().float()
        frames = F.interpolate(frames, size=(8 * h, 8 * h), mode="bilinear", align_corners=False)   # cv2.resize, v02:186
    elif os.path.exists(first_mp4):
        import numpy as np
        from hi3d_official_b200 import video_io
        fr = np.stack(video_io.read_video_frames(first_mp4)[:T], 0)
        frames = torch.from_numpy(fr).permute(0, 3, 1, 2).float().cuda() / 127.5 - 1.0
        frames = F.interpolate(frames, size=(8 * h, 8 * h), mode="bilinear", align_corners=False)
    elif params.synthetic:
        frames = torch.rand(T, 3, 8 * h, 8 * h, device="cuda") * 2 - 1
    else:
        raise SystemExit(f"{first} not found (run pipeline_i2v_eval_v01.py first) and --synthetic not given")
    if params.cond:
        d = torch.load(params.cond, map_location="cuda")
        c, uc = d["c"], d["uc"]
    elif params.towers:
        c, uc = cond_from_towers(model, frames.permute(1, 0, 2, 3).contiguous(), torch.load(params.towers), params.elevation, 2)
    elif params.synthetic:
        c, uc = synthetic_cond(2, T, h, "cuda", seed)
    else:
        raise SystemExit("the conditioner towers are outside the B200 hot path: pass --towers / --cond <file> or --synthetic")
    with torch.no_grad():
        init_latents = torch.randn(T, 4, h, h, device="cuda")                                      # v02:93
        z = torch.cat([model.encode_first_stage(frames[t:t + 1].half()) for t in range(T)], 0)     # v02:96-101
        out = model.sample_stage2(c, uc, init_latents, z.float())                                  # v02:103-137
    mp4 = save_frames(out, os.path.join(params.output_dir, "second_step_video"), "second")
    print(f"[hi3d-b200] wrote {T} frames {tuple(out.shape[1:])} to {mp4} (seed {seed})")


if __name__ == "__main__":
    main()
