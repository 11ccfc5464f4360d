#!/usr/bin/env python
"""bench.py -- Hi3D denoising hot path on B200.

One "step" = one orbital video of the workload: 25 Euler-EDM sampler steps of the CFG-batched VideoUNet
(N = 2 x 16 frames) followed by the AutoencoderKL decode of the 16 frames.  Metric = multi-view frames / s.

Default workload: BASELINE.json configs[2], second-stage 16 x 1024 x 1024 (latents 16 x 4 x 128 x 128, 17-channel UNet
input = [x | depth 9 | cond latent 4], v02 re-noise loop), fp16 (the reference's inference dtype and the parity dtype;
SURVEY F4) -- the largest single-GPU configuration and the shape the north-star target is stated on.  The stage-1 number
(configs[1], 16 x 512 x 512) is measured in the same N=1 run and reported under the extra key `stage1`
(`--stage 1` makes it the main line instead).
With --gpus N > 1 (torchrun) the default is `--shard frames` (configs[3], the north-star layout): ONE video whose 16 frames
are sharded over the ranks (strong scaling; K/V exchange before temporal attention, one-frame halo for the (3,1,1) convs,
(sum, sumsq) exchange for the (T,H,W) GroupNorm -- through peer memory over NVLink inside the consuming kernels, or NCCL
with HI3D_SHARD_EXCHANGE=nccl).  `--shard videos` = one video per GPU (configs[4], weak scaling, no data-path collective).
In frames mode the line also carries `shard_selfcheck` (max |err| of one sharded sampler step against the same step run
unsharded on the same GPU) and `exchange` (device time of the separable exchange launches of one UNet forward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--stage 1|2] [--shard videos|frames] [--impl reference]
                    [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (the decoded frames of rank 0's video) as DIR/frames.npy,
float32: whole when it fits in 64 MB (stage 1: 16 x 3 x 512 x 512), else a fixed sample (stage 2, see `dump_outputs`).
Inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.  The
GroupNorm statistics are accumulated with float atomics, so two runs agree to rounding, not bit for bit.

stdout carries exactly one line, the JSON (libraries that print to fd 1 are redirected to stderr).  Keys beyond the
contract: `unet_ms_per_sampler_step` (one eager UNet forward with the host kept ahead of the GPU = the cost of a sampler
step inside the graph), `kernel_breakdown` (CUDA events around every launch of one instrumented forward: per kernel class
ms / share / TFLOP/s / GB/s, the top GEMM shapes, and the sum of launches), `roofline` (all GEMM launches of that forward
against the measured sustained bf16 peak of MEASURED_PEAKS.json).

--impl reference times THE REFERENCE ITSELF -- the unmodified `sgm` modules staged byte-for-byte under oracle/_ref by
oracle/build_ref.py (kind "reference"; the oracle port only if that copy is absent) -- on the host cores, fp32, at the
config's OWN latent size: each bench "step" (a 25-step video) is sampled by real `EulerEDMSampler.sampler_step` calls (one
CFG-batched VideoUNet forward + guider + Euler update each; all 25 steps of a video cost the same) and reported as
16 frames / (25 x seconds per sampler step); no projection across shapes.  A real step takes minutes on a CPU, so the arm
is bounded by --ref-budget-s: it runs as many of the requested warm-up + timed sampler steps as fit and says how many.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "multi-view frames/sec (16f, 25-step EDM)"
T_FRAMES = 16
NUM_STEPS = 25


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------------------------
def workload(stage: int):
    if stage == 1:
        return dict(name="first-stage inference-v01 16x512x512, 25 EDM steps", h=64, cc=4, adm=768, max_scale=2.5)
    return dict(name="second-stage inference-v02 16x1024x1024 depth-concat, 25 EDM steps", h=128, cc=13, adm=512,
                max_scale=2.0)


def make_host_inputs(stage: int, seed: int, pin: bool):
    import torch
    wl = workload(stage)
    g = torch.Generator().manual_seed(1234 + seed)
    h = wl["h"]
    t = dict(randn=torch.randn(T_FRAMES, 4, h, h, generator=g),
             crossattn=torch.randn(1, 1, 1024, generator=g),
             vector=torch.randn(1, wl["adm"], generator=g),
             concat=(torch.randn(T_FRAMES, wl["cc"], h, h, generator=g) * 0.18).half())
    if stage == 2:
        t["z"] = torch.randn(T_FRAMES, 4, h, h, generator=g) * 0.18
    if pin:
        t = {k: v.pin_memory() for k, v in t.items()}
    return t


def to_cond(dev_t):
    import torch
    c = dict(crossattn=dev_t["crossattn"], vector=dev_t["vector"], concat=dev_t["concat"])
    uc = dict(crossattn=torch.zeros_like(c["crossattn"]), vector=c["vector"], concat=torch.zeros_like(c["concat"]))
    return c, uc


def run_video(model, stage: int, dev_t, shard=None):
    c, uc = to_cond(dev_t)
    if stage == 1:
        return model.sample_stage1(c, uc, dev_t["randn"].clone(), shard=shard)
    return model.sample_stage2(c, uc, dev_t["randn"].clone(), dev_t["z"], shard=shard)


def shard_frames(t: dict, rank: int, world: int) -> dict:
    """This rank's frames of the per-frame tensors (BASELINE configs[3]: one video, frames sharded over GPUs)."""
    tl = T_FRAMES // world
    sl = slice(rank * tl, (rank + 1) * tl)
    return {k: (v[sl].contiguous() if v.shape[0] == T_FRAMES else v) for k, v in t.items()}


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full` capture
# (not measurable live): mean over the 10 hi3d_gemm_tc5 launches of input block 1 (64x64 level: conv3x3, temporal conv,
# proj_in, qkv, attention out, GEGLU, ff2 ...), each 84-420 MB algorithmic.  Stage 2 was not captured.
NCU_GEMM_TRAFFIC = {1: 292.8e6, 2: 1163.7e6}
NCU_GEMM_TRAFFIC_NOTE = {
    1: ("bytes per launch, mean of the 10 top-level GEMM launches in profiles/r01_ncu_full_stage1_final.txt "
        "(ncu --set full, caches flushed per pass); `achieved` averages all 300 GEMM launches of a forward"),
    2: ("dram__bytes_read.sum + dram__bytes_write.sum per launch, mean of the 13 top-level (128x128 latent) GEMM launches in "
        "profiles/r02_ncu_full_stage2.txt (ncu --set full, caches flushed per pass; algorithmic bytes of the same launches: "
        "A + output + residual = 0.67-1.7 GB); `achieved` averages all 300 GEMM launches of a forward"),
}


def kernel_breakdown(model, stage: int, dev_t, peaks):
    """One extra, instrumented sampler step: CUDA events around every launch of the UNet plan on the launching
    stream -> per kernel-class time, algorithmic FLOPs / bytes, achieved rate."""
    import torch
    from hi3d_official_b200 import ops
    unet = model.model.diffusion_model
    wl = workload(stage)
    plan = unet.get_plan(2 * T_FRAMES, wl["h"], wl["h"], T_FRAMES)
    recs = []
    # queue ~60 ms of spinning first so the host gets ahead of the GPU: otherwise the short kernels (norms, small GEMMs)
    # are bracketed together with the idle time the GPU spends waiting for their launch
    torch.cuda._sleep(int(1.2e8))
    for s in plan.steps:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); s(); e1.record()
        recs.append((s, e0, e1))
    torch.cuda.synchronize()
    # the whole UNet forward back to back (host far ahead of the GPU) = what one sampler step costs inside the graph
    torch.cuda._sleep(int(4e7))
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(3):
        for s in plan.steps:
            s()
    f1.record()
    torch.cuda.synchronize()
    fwd_ms = f0.elapsed_time(f1) / 3
    cls = {}
    for s, e0, e1 in recs:
        ms = e0.elapsed_time(e1)
        if isinstance(s, ops.Gemm):
            k, fl, by = "gemm(conv/linear)", s.flops, 0.0
        else:
            k, fl, by = getattr(s, "kind", "other"), getattr(s, "flops", 0.0), getattr(s, "bytes", 0.0)
        d = cls.setdefault(k, dict(ms=0.0, launches=0, flops=0.0, bytes=0.0))
        d["ms"] += ms; d["launches"] += 1; d["flops"] += fl; d["bytes"] += by
    tot = sum(d["ms"] for d in cls.values())
    # per GEMM shape (rows mode, M, N, K, activation): where the implicit-GEMM time goes
    shapes = {}
    for s, e0, e1 in recs:
        if isinstance(s, ops.Gemm):
            pp = s.p
            key = f"mode{pp.mode} M={pp.M} N={pp.N} K={pp.K} act={pp.act}" + (" up" if pp.out_up else "") + \
                  (" s2" if pp.stride == 2 else "")
            d = shapes.setdefault(key, dict(ms=0.0, launches=0, flops=0.0))
            d["ms"] += e0.elapsed_time(e1); d["launches"] += 1; d["flops"] += s.flops
    top = sorted(shapes.items(), key=lambda kv: -kv[1]["ms"])[:14]
    out = {}
    out["gemm_shapes_top"] = {k: dict(ms=round(d["ms"], 3), launches=d["launches"], tflops=round(d["flops"] / d["ms"] / 1e9, 1))
                              for k, d in top}
    for k, d in cls.items():
        out[k] = dict(ms=round(d["ms"], 3), share=round(d["ms"] / tot, 4), launches=d["launches"])
        if d["flops"]:
            out[k]["tflops"] = round(d["flops"] / d["ms"] / 1e9, 1)
        if d["bytes"]:
            out[k]["gbs"] = round(d["bytes"] / d["ms"] / 1e6, 1)
            out[k]["hbm_frac"] = round(d["bytes"] / d["ms"] / 1e6 / peaks["hbm"], 4)
    g = cls.get("gemm(conv/linear)")
    roof = None
    if g:
        ach = g["flops"] / g["ms"] / 1e9
        roof = dict(bound="tensor", kernel="hi3d_gemm (implicit-GEMM conv/linear, all launches of one UNet step)",
                    achieved=round(ach, 1), peak=peaks["tf_sust"], unit="TFLOP/s", frac=round(ach / peaks["tf_sust"], 4),
                    peak_source=f"{peaks['src']} bf16_tflops_sustained", traffic=NCU_GEMM_TRAFFIC.get(stage),
                    traffic_note=NCU_GEMM_TRAFFIC_NOTE.get(stage),
                    flops_per_step=g["flops"], avg_launch_ms=round(g["ms"] / g["launches"], 4))
    out["sum_of_launches_ms"] = round(tot, 3)
    return out, roof, fwd_ms


class ReferenceCPU:
    """The reference's own CPU path for one sampler step, on the host cores (fp32): the unmodified sgm modules
    (`VideoUNet`, `OpenAIWrapper`, `Denoiser`, `EulerEDMSampler` + `LinearPredictionGuider`) from /root/reference or its
    byte-for-byte staged copy oracle/_ref (kind "reference"); only when neither exists, the oracle port (kind "port").
    Weights: synthetic values of the bench's distribution (timing only; parity is pinned elsewhere)."""

    def __init__(self, stage: int, threads: int):
        import torch
        self.stage, self.threads = stage, threads
        torch.set_num_threads(threads)
        from hi3d_official_b200 import configs, spec
        kw = dict(configs.UNET_STAGE1 if stage == 1 else configs.UNET_STAGE2)
        self.wl = workload(stage)
        self.kind = "port"
        self.spec, self.kw = spec, kw
        try:
            from oracle import ref_import as R
            if R.available():
                R.setup()
                self.kind = "reference"
                self.R = R
        except Exception as e:      # noqa: BLE001
            print(f"[bench] reference modules unavailable ({e}); timing the oracle port", file=sys.stderr)
        if self.kind == "reference":
            from sgm.modules.diffusionmodules.video_model import VideoUNet
            kw2 = dict(kw, use_checkpoint=False, spatial_transformer_attn_type="softmax")     # SURVEY F6: xformers absent
            with torch.device("meta"):
                net = VideoUNet(**kw2)
            net = net.to_empty(device="cpu").eval()
            self._fill(net)
            self.net = R.wrap(net)
            self.denoiser = R.build_denoiser()
            self.sampler = R.build_sampler(num_steps=NUM_STEPS, max_scale=self.wl["max_scale"], num_frames=T_FRAMES, device="cpu")
            self.source = "oracle/_ref (staged copy of the unmodified reference)" if R.is_staged_copy() else R.REF_ROOT
        else:
            cfg = spec.UNetConfig.from_kwargs(**kw)
            self.sd = spec.synth_state_dict(spec.unet_param_shapes(cfg), seed=1)
            self.source = "oracle/hi3d_oracle.py (port)"

    def _fill(self, net):
        """Synthetic weights with the per-key scale of spec.synth_state_dict from one 16 M-element random block (a full
        per-key draw of 1.5 B values costs ~40 s of host time on the billed GPU box and changes no timing)."""
        import torch
        g = torch.Generator().manual_seed(7)
        block = torch.randn(1 << 24, generator=g)
        with torch.no_grad():
            for k, p in net.state_dict().items():
                n = p.numel()
                reps = (n + block.numel() - 1) // block.numel()
                x = (block if reps == 1 else block.repeat(reps))[:n].view(p.shape)
                p.copy_(self.spec._synth_rule(k, x))

    def inputs(self, latent: int):
        import torch
        g = torch.Generator().manual_seed(0)
        wl = self.wl
        x = torch.randn(T_FRAMES, 4, latent, latent, generator=g)
        c = dict(crossattn=torch.randn(1, 1, 1024, generator=g), vector=torch.randn(1, wl["adm"], generator=g),
                 concat=torch.randn(T_FRAMES, wl["cc"], latent, latent, generator=g) * 0.18)
        uc = dict(crossattn=torch.zeros(1, 1, 1024), vector=c["vector"], concat=torch.zeros_like(c["concat"]))
        return x, c, uc

    def sampler_step(self, x, c, uc, sigma=10.0, sigma_next=8.0) -> float:
        """One real sampler step (pipeline_i2v_eval_v01.py:85-92 closure + sampling.py:93-107); returns seconds."""
        import torch
        t0 = time.time()
        with torch.no_grad():
            if self.kind == "reference":
                kw = dict(image_only_indicator=torch.zeros(2, T_FRAMES), num_video_frames=T_FRAMES)

                def denoiser(inp, sig, cc):
                    return self.denoiser(self.net, inp, sig, cc, **kw)
                s_in = x.new_ones([x.shape[0]])
                out = self.sampler.sampler_step(s_in * sigma, s_in * sigma_next, denoiser, x, c, uc, gamma=0.0)
            else:
                from oracle import hi3d_oracle as O
                out = O.euler_step(self.sd, x, sigma, sigma_next, c, uc, O.guider_scale(T_FRAMES, self.wl["max_scale"]),
                                   num_video_frames=T_FRAMES)
        assert bool(torch.isfinite(out).all())
        return time.time() - t0


def host_threads() -> int:
    """Threads for the CPU arm: the physical cores this process may use, capped at 64 (oneDNN stops scaling well before
    that on these shapes and more threads only oversubscribe)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    phys = max(1, n // 2) if n > 16 else n          # SMT siblings do not help fp32 GEMM / conv
    return max(1, min(phys, int(os.environ.get("HI3D_CPU_THREADS", 64))))


def unet_step_flops(stage: int, latent: int) -> float:
    """Algorithmic FLOPs of one CFG-batched UNet forward (GEMM + attention cores), from the plan description."""
    # analytic: use the same counting as _Plan.flops without touching the GPU
    from hi3d_official_b200 import configs, spec
    kw = configs.UNET_STAGE1 if stage == 1 else configs.UNET_STAGE2
    cfg = spec.UNetConfig.from_kwargs(**kw)
    plan = spec.unet_plan(cfg)
    N, T = 2 * T_FRAMES, T_FRAMES
    fl = 0.0
    for blk in plan.input_blocks + [plan.middle] + plan.output_blocks:
        for L in blk:
            hw = (latent // L.ds) ** 2
            M = N * hw
            if L.kind in ("conv_in", "down", "up"):
                mo = M // 4 if L.kind == "down" else (M * 4 if L.kind == "up" else M)
                fl += 2.0 * mo * L.cout * 9 * L.cin
            elif L.kind == "res":
                fl += 2.0 * M * L.cout * 9 * L.cin + 2.0 * M * L.cout * 9 * L.cout
                if L.cin != L.cout:
                    fl += 2.0 * M * L.cout * L.cin
                fl += 2 * (2.0 * M * L.cout * 3 * L.cout)
            elif L.kind == "attn":
                C = L.cin
                per_blk = 2.0 * M * C * (3 * C + C + 8 * C + 4 * C)       # qkv, out, ff1, ff2
                fl += 2.0 * M * C * C * 2                                 # proj_in / proj_out
                fl += per_blk + per_blk + 2.0 * M * C * 12 * C            # spatial, temporal, + ff_in
                fl += 4.0 * N * hw * hw * C + 4.0 * N * hw * T * C        # attention cores
    return fl


DUMP_BYTES = 64 * 10 ** 6      # all of what --dump-outputs writes


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each array as <out_dir>/<name>.npy in float32.  One whose float32 size exceeds its share of DUMP_BYTES is
    written as a fixed sample instead: the flattened array at the first k indices of
    numpy.random.RandomState(0).permutation(numel), sorted (a 1-D array; RandomState keeps its stream across numpy
    versions)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.float().numpy()
        what = f"{a.shape}"
        if a.nbytes > share:
            k = (share - 4096) // 4                    # leave room for the .npy header
            idx = np.sort(np.random.RandomState(0).permutation(a.size)[:k])
            a = a.reshape(-1)[idx]
            what = f"a fixed sample of {k} of the {t.numel()} elements of {tuple(t.shape)}"
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        print(f"[bench] --dump-outputs: {name}.npy = {what}", file=sys.stderr)


# ------------------------------------------------------------------------------------------------------------------
def measure(model, stage, engine, rank, world, local, dev, steps, warmup, frames_mode, dist, want_breakdown, peaks,
            keep_output=False):
    """Warm up, time `steps` videos device-resident and e2e; returns a dict of raw results (rank 0 has everything).
    keep_output: also return what the last timed resident step computed, on the host (`output`)."""
    import torch
    from hi3d_official_b200 import _native
    wl = workload(stage)
    shard = (rank, world) if frames_mode else None
    host = make_host_inputs(stage, seed=0 if frames_mode else rank, pin=True)
    if frames_mode:
        host = {k: v.pin_memory() for k, v in shard_frames(host, rank, world).items()}
    dev_t = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
    n_local = T_FRAMES // world if frames_mode else T_FRAMES
    out_host = torch.empty(n_local, 3, wl["h"] * 8, wl["h"] * 8, dtype=torch.float16).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = out_host.numel() * out_host.element_size()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _native.launch_count()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), _native.launch_count() - l0

    last = [None]

    def step_resident():
        out = run_video(model, stage, dev_t, shard)
        if keep_output:
            last[0] = out

    def step_e2e():
        d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        frames = run_video(model, stage, d, shard)
        out_host.copy_(frames, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(max(warmup, 3)):
        step_resident()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms, launches = timed(step_resident, steps)
    clk = clocks.stop() if rank == 0 else None
    output = last[0].cpu() if keep_output else None      # before the e2e steps can reuse its memory
    step_e2e()
    ms_e2e, _ = timed(step_e2e, steps)
    res = dict(ms=ms, ms_e2e=ms_e2e, launches=launches, clocks=clk, h2d=h2d, d2h=d2h, breakdown=None, roof=None, unet_ms=None,
               output=output)
    if rank == 0 and want_breakdown and not frames_mode:
        res["breakdown"], res["roof"], res["unet_ms"] = kernel_breakdown(model, stage, dev_t, peaks)
    if frames_mode:
        res["selfcheck"], res["exchange"] = shard_selfcheck(model, stage, rank, world, dev, dist)
    return res


def shard_selfcheck(model, stage, rank, world, dev, dist):
    """(i) One fused sampler step of the frame-sharded plan against the SAME step run unsharded on this GPU (all 16 frames,
    same weights / inputs): max |err| over this rank's frames, max over ranks.  (ii) device time of the separable exchange
    launches (kind 'exchange' / 'nccl') of one eager UNet forward of the sharded plan, max over ranks."""
    import torch
    full = make_host_inputs(stage, seed=0, pin=False)
    full = {k: v.to(dev) for k, v in full.items()}
    c, uc = to_cond(full)
    T = T_FRAMES
    tl = T // world
    sl = slice(rank * tl, (rank + 1) * tl)
    smp = model.sampler
    sig, sig_n = 10.0, 8.0
    x = (full["randn"] * (1.0 + sig ** 2) ** 0.5).contiguous()
    den_full = model.bind_denoiser(image_only_indicator=None, num_video_frames=T)
    s16 = torch.full((T,), sig, device=dev)
    st = smp._fused_state(den_full, x, c, uc, refresh=True)
    ref = st.step(x, s16, s16 * (sig_n / sig)).clone()
    cl = dict(c, concat=c["concat"][sl].contiguous())
    ucl = dict(uc, concat=uc["concat"][sl].contiguous())
    den_sh = model.bind_denoiser(shard=(rank, world), image_only_indicator=None, num_video_frames=T)
    xs = x[sl].contiguous()
    sl_sig = torch.full((tl,), sig, device=dev)
    st2 = smp._fused_state(den_sh, xs, cl, ucl, refresh=True)
    got = st2.step(xs, sl_sig, sl_sig * (sig_n / sig)).clone()
    torch.cuda.synchronize()
    err = torch.tensor([float((got - ref[sl]).abs().max())], device=dev)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    check = {"max_abs_err_vs_unsharded_step": float(err.item()), "ref_mean_abs": float(ref.abs().mean()),
             "sigma": sig, "note": "one fused Euler step, sharded plan vs the unsharded plan on the same GPU"}
    # exchange launches of one eager forward (all ranks execute every launch in the same order; events only around them)
    plan = st2.plan
    recs = []
    dist.barrier()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for s_ in plan.steps:
        if getattr(s_, "kind", "") in ("nccl", "exchange"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); s_(); e1.record()
            recs.append((e0, e1))
        else:
            s_()
    f1.record()
    torch.cuda.synchronize()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in recs), f0.elapsed_time(f1)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    exch = {"exchange_launches_per_unet_forward": len(recs), "exchange_ms_per_unet_forward": round(float(t[0]), 3),
            "eager_unet_forward_ms": round(float(t[1]), 3), "mode": getattr(plan, "exchange_mode", "nccl"),
            "note": "separable exchange launches only (NCCL calls / flag barriers); peer-memory loads fused into the temporal "
                    "attention / conv / GroupNorm kernels are part of those kernels' time"}
    return check, exch


def reference_arm(args, wl, config, emit):
    """`--impl reference`: real sampler steps of the reference's CPU path at the config's own latent size."""
    threads = host_threads()
    t_build = time.time()
    ref = ReferenceCPU(args.stage, threads)
    lat = wl["h"]
    if args.ref_latent:
        lat = args.ref_latent
        config = dict(config, reference_latent_override=lat)
    x, c, uc = ref.inputs(lat)
    t_build = time.time() - t_build
    t_start = time.time()
    want = args.warmup + args.steps
    times = []
    while len(times) < want:
        times.append(ref.sampler_step(x, c, uc))
        left = args.ref_budget_s - (time.time() - t_start)
        if left < 1.15 * max(times):            # the next step would overrun the budget
            break
    n_warm = min(args.warmup, max(0, len(times) - 1))          # at least one timed step
    timed = times[n_warm:]
    t = sum(timed) / len(timed)
    fps = T_FRAMES / (NUM_STEPS * t)
    sample = (f"{len(timed)} timed + {n_warm} warm-up REAL sampler steps (of {args.steps} + {args.warmup} requested; bounded by "
              f"--ref-budget-s {args.ref_budget_s:.0f}) of {ref.source}: CFG-batched full-width VideoUNet forward + guider + Euler, "
              f"fp32, {lat}x{lat} latents, {threads} threads = {t:.1f} s per sampler step (each: "
              f"{', '.join(f'{v:.1f}' for v in times)}); a video = 25 such steps; VAE decode not included; model build {t_build:.0f} s untimed")
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": NUM_STEPS * t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": config,
            "sampler_steps_timed": len(timed), "sampler_step_s": t,
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": ref.kind, "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--stage", type=int, default=2, choices=(1, 2))
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--engine", default=os.environ.get("HI3D_ENGINE", "tc5"), choices=("mma", "tc5"))
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--shard", default=None, choices=("videos", "frames"),
                    help="N > 1: 'frames' (default) = ONE video with its 16 frames sharded over the GPUs (strong scaling; K/V "
                         "+ halo + GN-statistics exchange per temporal layer); 'videos' = one video per GPU (weak scaling)")
    ap.add_argument("--cpu-latent", type=int, default=48,
                    help="latent size of the bounded cpu_baseline sample of the main arm (one real reference sampler step)")
    ap.add_argument("--ref-budget-s", type=float, default=float(os.environ.get("HI3D_REF_BUDGET_S", 300)),
                    help="--impl reference: wall-clock budget for the real full-size sampler steps")
    ap.add_argument("--no-stage1", action="store_true", help="skip the extra stage-1 measurement of the N=1 stage-2 run")
    ap.add_argument("--ref-latent", type=int, default=0,
                    help="TESTS ONLY (--impl reference): latent size override so the CPU suite finishes in seconds; the line "
                         "then says so in config.reference_latent_override and is not a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path, not --impl reference")
    # stdout carries exactly ONE line, the JSON: anything a library writes to fd 1 in between (NCCL prints its version
    # banner there) goes to stderr instead
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(_real_stdout, (json.dumps(line) + "\n").encode())
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    wl = workload(args.stage)
    shard_mode = args.shard or ("frames" if world > 1 else "videos")
    frames_mode = shard_mode == "frames" and world > 1
    config = {"workload": wl["name"], "frames": T_FRAMES, "sampler_steps": NUM_STEPS, "latent": [T_FRAMES, 4, wl["h"], wl["h"]],
              "cfg_batch": 2 * T_FRAMES, "vae_decode_in_step": True,
              "parallelism": (f"frames of ONE video sharded over {world} GPUs ({T_FRAMES // max(world, 1)} per GPU)" if frames_mode
                              else f"dp{world} (one video per GPU)"),
              "l2": "activations >> L2 (UNet working set > 1 GB per step); no flush needed"}

    if args.impl == "reference":
        if rank != 0:
            return
        # the CPU arm always describes the single-video workload of the config (no GPUs involved)
        reference_arm(args, wl, config, emit)
        return

    import torch
    import torch.distributed as dist
    from hi3d_official_b200 import configs, spec
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout = the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    if frames_mode and T_FRAMES % world:
        raise SystemExit(f"--shard frames needs 16 % world == 0, got {world}")
    peaks = _peaks()

    def build(stage):
        m = configs.build_engine(stage, device=dev)
        spec.synth_fill_(m, seed=0, fast=True)
        m.model.diffusion_model.set_engine(args.engine)
        m.first_stage_model.set_engine(args.engine)
        return m

    model = build(args.stage)
    r = measure(model, args.stage, args.engine, rank, world, local, dev, args.steps, args.warmup, frames_mode, dist,
                not args.no_breakdown, peaks, keep_output=bool(args.dump_outputs) and rank == 0)
    if r["output"] is not None:
        dump_outputs(args.dump_outputs, {"frames": r.pop("output")})
    stage1 = None
    if rank == 0 and world == 1 and args.stage == 2 and not args.no_stage1:
        del model
        torch.cuda.empty_cache()
        k1 = max(1, min(args.steps, 5))
        m1 = build(1)
        r1 = measure(m1, 1, args.engine, 0, 1, local, dev, k1, 3, False, dist, not args.no_breakdown, peaks)
        stage1 = {"workload": workload(1)["name"], "value": T_FRAMES * k1 / (r1["ms"] / 1e3), "unit": "frames/s", "steps": k1,
                  "warmup": 3, "ms_per_step": r1["ms"] / k1, "e2e": T_FRAMES * k1 / (r1["ms_e2e"] / 1e3),
                  "unet_ms_per_sampler_step": r1["unet_ms"], "roofline": r1["roof"], "kernel_breakdown": r1["breakdown"]}
        del m1
        torch.cuda.empty_cache()
    cpu_b = None
    if rank == 0 and world == 1 and not os.environ.get("HI3D_SKIP_CPU_BASELINE"):
        lat = min(args.cpu_latent, wl["h"])
        threads = host_threads()
        ref = ReferenceCPU(args.stage, threads)
        x, c, uc = ref.inputs(lat)
        t = ref.sampler_step(x, c, uc)
        ratio = unet_step_flops(args.stage, wl["h"]) / unet_step_flops(args.stage, lat)
        cpu_b = {"value": T_FRAMES / (NUM_STEPS * t * ratio), "unit": "frames/s", "cores": threads, "kind": ref.kind,
                 "sample": f"ONE real sampler step of {ref.source} (full-width stage-{args.stage} VideoUNet, CFG batch 32, fp32, "
                           f"{threads} threads) at {lat}x{lat} latents = {t:.1f} s" +
                           (f", scaled to {wl['h']}x{wl['h']} by the UNet FLOP ratio {ratio:.2f}" if ratio != 1.0 else "") +
                           " x 25 steps per video; `bench.py --impl reference` times the full size"}
    if rank == 0:
        videos = 1 if frames_mode else world
        ms, ms_e2e = r["ms"], r["ms_e2e"]
        fps = T_FRAMES * args.steps * videos / (ms / 1e3)
        fps_e2e = T_FRAMES * args.steps * videos / (ms_e2e / 1e3)
        line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if frames_mode else "weak",
                "vs_baseline": None, "dtype": "fp16", "data": "synthetic", "config": config, "engine": args.engine,
                "unet_ms_per_sampler_step": r["unet_ms"], "clocks": r["clocks"],
                "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]},
                "gpu_launches": r["launches"], "roofline": r["roof"], "kernel_breakdown": r["breakdown"], "cpu_baseline": cpu_b}
        if frames_mode:
            line["shard_selfcheck"], line["exchange"] = r["selfcheck"], r["exchange"]
        if stage1 is not None:
            line["stage1"] = stage1
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except SystemExit:
        raise
    except BaseException:          # a failed rank must not leave its peers waiting in a collective until the NCCL timeout
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
