"""Cost of the deterministic mode (HI3D_DETERMINISTIC=1): the full-width UNet forward at the stage-1 (64 x 64 latents) and
stage-2 (128 x 128) shapes, CFG batch 32 (16 frames), timed with CUDA events in both modes, alternating mode by mode in
one process on the same build and weights, plus the library launches per forward.  The card's name and power limit are
read in the same run and stored with the numbers.

    python tools/deterministic_cost.py --out profiles/r03_deterministic_cost.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hi3d_official_b200 import _native, configs, spec  # noqa: E402
from hi3d_official_b200.unet import VideoUNet  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    cfg = spec.UNetConfig.from_kwargs(**configs.UNET_STAGE1)
    net = VideoUNet(**configs.UNET_STAGE1)
    net.load_state_dict(spec.synth_state_dict(spec.unet_param_shapes(cfg), seed=1), strict=True)
    net = net.cuda().half()
    T, N = 16, 32
    res = {"card": card(), "torch": torch.__version__, "shapes": {}}
    for name, hw in (("stage1_64x64", 64), ("stage2_128x128", 128)):
        g = torch.Generator().manual_seed(0)
        x = torch.randn(N, 8, hw, hw, generator=g).cuda()
        ctx = torch.randn(N // T, 1, 1024, generator=g).cuda()
        y = torch.randn(N // T, 768, generator=g).cuda()
        t = torch.full((N,), 0.7, device="cuda")
        times = {"0": [], "1": []}
        launches, outs = {}, {}
        for mode in ("0", "1"):                       # build both plans and warm them up
            os.environ["HI3D_DETERMINISTIC"] = mode
            for _ in range(2):
                outs[mode] = net(x, timesteps=t, context=ctx, y=y, num_video_frames=T)
            torch.cuda.synchronize()
            c0 = _native.launch_count()
            net(x, timesteps=t, context=ctx, y=y, num_video_frames=T)
            torch.cuda.synchronize()
            launches[mode] = _native.launch_count() - c0
        for _ in range(a.rounds):
            for mode in ("0", "1"):
                os.environ["HI3D_DETERMINISTIC"] = mode
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.reps):
                    net(x, timesteps=t, context=ctx, y=y, num_video_frames=T)
                e1.record()
                torch.cuda.synchronize()
                times[mode].append(e0.elapsed_time(e1) / a.reps)
        d, m = statistics.median(times["0"]), statistics.median(times["1"])
        res["shapes"][name] = {
            "unet_forward_ms": {"default": d, "deterministic": m, "all_rounds": times},
            "deterministic_over_default": m / d,
            "launches_per_forward": launches,
            "max_abs_diff_default_vs_deterministic": float((outs["0"].float() - outs["1"].float()).abs().max()),
        }
        print(name, json.dumps(res["shapes"][name]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
