"""Sampler-side operator surface of the reference, same names and call signatures:

  EDMDiscretization            sgm/modules/diffusionmodules/discretizer.py:17-39
  VScalingWithEDMcNoise (+EDM/Eps/V scalings)   denoiser_scaling.py:11-59
  Denoiser                     denoiser.py:12-39
  IdentityWrapper / OpenAIWrapper   wrappers.py:8-34
  IdentityGuider / VanillaCFG / LinearPredictionGuider   guiders.py:24-99
  BaseDiffusionSampler / EDMSampler / EulerEDMSampler (+ Hi3D's step_call)   sampling.py:21-147,228-232

Two execution paths with identical results:
  * generic: `denoiser` is any Python callable (x, sigma, cond) -> denoised, exactly like the reference; the
    few elementwise ops on the (16, 4, h, w) fp32 sampler state are torch glue around whatever the callable does;
  * fused (the product path): when the callable is a `FusedDenoiser` binding (Denoiser + OpenAIWrapper(VideoUNet)),
    one Euler step is  hi3d_sampler_pre -> VideoUNet launch plan -> hi3d_sampler_post  with no host sync,
    no torch math and the step-invariant conditioning computed once per video.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import _native, ops
from .unet import CIN_PAD, VideoUNet
from .util import append_dims, append_zero, default, instantiate_from_config

OPENAIUNETWRAPPER = "sgm.modules.diffusionmodules.wrappers.OpenAIWrapper"


# ------------------------------------------------------------------------------------------------------------
# discretisation / scalings
# ------------------------------------------------------------------------------------------------------------
class Discretization:
    def __call__(self, n, do_append_zero=True, device="cpu", flip=False):
        sigmas = self.get_sigmas(n, device=device)
        sigmas = append_zero(sigmas) if do_append_zero else sigmas
        return sigmas if not flip else torch.flip(sigmas, (0,))

    def get_sigmas(self, n, device):
        raise NotImplementedError


class EDMDiscretization(Discretization):
    def __init__(self, sigma_min=0.002, sigma_max=80.0, rho=7.0):
        self.sigma_min, self.sigma_max, self.rho = sigma_min, sigma_max, rho

    def get_sigmas(self, n, device="cpu"):
        ramp = torch.linspace(0, 1, n, device=device)
        min_inv_rho = self.sigma_min ** (1 / self.rho)
        max_inv_rho = self.sigma_max ** (1 / self.rho)
        return (max_inv_rho + ramp * (min_inv_rho - max_inv_rho)) ** self.rho


class EDMScaling:
    def __init__(self, sigma_data: float = 0.5):
        self.sigma_data = sigma_data

    def __call__(self, sigma):
        c_skip = self.sigma_data ** 2 / (sigma ** 2 + self.sigma_data ** 2)
        c_out = sigma * self.sigma_data / (sigma ** 2 + self.sigma_data ** 2) ** 0.5
        c_in = 1 / (sigma ** 2 + self.sigma_data ** 2) ** 0.5
        return c_skip, c_out, c_in, 0.25 * sigma.log()


class EpsScaling:
    def __call__(self, sigma):
        return torch.ones_like(sigma), -sigma, 1 / (sigma ** 2 + 1.0) ** 0.5, sigma.clone()


class VScaling:
    def __call__(self, sigma):
        return 1.0 / (sigma ** 2 + 1.0), -sigma / (sigma ** 2 + 1.0) ** 0.5, 1.0 / (sigma ** 2 + 1.0) ** 0.5, sigma.clone()


class VScalingWithEDMcNoise:
    def __call__(self, sigma):
        c_skip = 1.0 / (sigma ** 2 + 1.0)
        c_out = -sigma / (sigma ** 2 + 1.0) ** 0.5
        c_in = 1.0 / (sigma ** 2 + 1.0) ** 0.5
        c_noise = 0.25 * sigma.log()
        return c_skip, c_out, c_in, c_noise


# ------------------------------------------------------------------------------------------------------------
# denoiser + wrappers
# ------------------------------------------------------------------------------------------------------------
class Denoiser(nn.Module):
    def __init__(self, scaling_config: Dict):
        super().__init__()
        self.scaling = instantiate_from_config(scaling_config)

    def possibly_quantize_sigma(self, sigma):
        return sigma

    def possibly_quantize_c_noise(self, c_noise):
        return c_noise

    def forward(self, network: nn.Module, input: torch.Tensor, sigma: torch.Tensor, cond: Dict,
                **additional_model_inputs) -> torch.Tensor:
        sigma = self.possibly_quantize_sigma(sigma)
        sigma_shape = sigma.shape
        sigma = append_dims(sigma, input.ndim)
        c_skip, c_out, c_in, c_noise = self.scaling(sigma)
        c_noise = self.possibly_quantize_c_noise(c_noise.reshape(sigma_shape))
        return network(input * c_in, c_noise, cond, **additional_model_inputs) * c_out + input * c_skip


class IdentityWrapper(nn.Module):
    def __init__(self, diffusion_model, compile_model: bool = False):
        super().__init__()
        if compile_model:
            raise NotImplementedError("torch.compile is not part of the B200 path (explicit kernels + CUDA graphs)")
        self.diffusion_model = diffusion_model

    def forward(self, *args, **kwargs):
        return self.diffusion_model(*args, **kwargs)


class OpenAIWrapper(IdentityWrapper):
    def forward(self, x: torch.Tensor, t: torch.Tensor, c: dict, **kwargs) -> torch.Tensor:
        x = torch.cat((x, c.get("concat", torch.Tensor([]).type_as(x)).to(x.dtype)), dim=1)
        return self.diffusion_model(x, timesteps=t, context=c.get("crossattn", None), y=c.get("vector", None), **kwargs)


# ------------------------------------------------------------------------------------------------------------
# guiders
# ------------------------------------------------------------------------------------------------------------
class IdentityGuider:
    def __call__(self, x, sigma):
        return x

    def prepare_inputs(self, x, s, c, uc):
        return x, s, {k: c[k] for k in c}


class VanillaCFG:
    def __init__(self, scale: float):
        self.scale = scale

    def __call__(self, x, sigma):
        x_u, x_c = x.chunk(2)
        return x_u + self.scale * (x_c - x_u)

    def prepare_inputs(self, x, s, c, uc):
        c_out = dict()
        for k in c:
            if k in ["vector", "crossattn", "concat"]:
                c_out[k] = torch.cat((uc[k], c[k]), 0)
            else:
                assert c[k] == uc[k]
                c_out[k] = c[k]
        return torch.cat([x] * 2), torch.cat([s] * 2), c_out


class LinearPredictionGuider:
    def __init__(self, max_scale: float, num_frames: int, min_scale: float = 1.0,
                 additional_cond_keys: Optional[Union[List[str], str]] = None):
        self.min_scale, self.max_scale, self.num_frames = min_scale, max_scale, num_frames
        self.scale = torch.linspace(min_scale, max_scale, num_frames).unsqueeze(0)
        additional_cond_keys = default(additional_cond_keys, [])
        if isinstance(additional_cond_keys, str):
            additional_cond_keys = [additional_cond_keys]
        self.additional_cond_keys = additional_cond_keys

    def __call__(self, x: torch.Tensor, sigma: torch.Tensor) -> torch.Tensor:
        x_u, x_c = x.chunk(2)
        T = self.num_frames
        x_u = x_u.reshape(-1, T, *x_u.shape[1:])
        x_c = x_c.reshape(-1, T, *x_c.shape[1:])
        scale = append_dims(self.scale.expand(x_u.shape[0], T), x_u.ndim).to(x_u.device)
        out = x_u + scale * (x_c - x_u)
        return out.reshape(-1, *out.shape[2:])

    def prepare_inputs(self, x, s, c, uc) -> Tuple[torch.Tensor, torch.Tensor, dict]:
        c_out = dict()
        for k in c:
            if k in ["vector", "crossattn", "concat"] + self.additional_cond_keys:
                c_out[k] = torch.cat((uc[k], c[k]), 0)
            else:
                assert c[k] == uc[k]
                c_out[k] = c[k]
        return torch.cat([x] * 2), torch.cat([s] * 2), c_out


# ------------------------------------------------------------------------------------------------------------
# fused binding
# ------------------------------------------------------------------------------------------------------------
class FusedDenoiser:
    """The pipelines' closure `lambda input, sigma, c: model.denoiser(model.model, input, sigma, c, **kw)`
    (pipeline_i2v_eval_v01.py:85-88) as an inspectable object, so the sampler can run the fused B200 step.
    Calling it behaves exactly like the closure (generic path)."""

    def __init__(self, denoiser: Denoiser, network: nn.Module, shard: Optional[Tuple[int, int]] = None,
                 **additional_model_inputs):
        self.denoiser, self.network, self.kwargs = denoiser, network, additional_model_inputs
        # shard = (rank, world): the caller passes only this rank's frames of x / cond['concat'] (frame sharding over
        # GPUs, SURVEY 8e); num_video_frames stays the GLOBAL frame count
        self.shard = None if shard is None or shard[1] == 1 else (int(shard[0]), int(shard[1]))

    def __call__(self, input, sigma, c):
        if self.shard is not None:
            raise NotImplementedError("a frame-sharded FusedDenoiser can only be evaluated by the fused Euler step "
                                      "(the generic closure has no cross-rank exchanges)")
        return self.denoiser(self.network, input, sigma, c, **self.kwargs)

    def fusable(self) -> bool:
        return (isinstance(self.denoiser.scaling, VScalingWithEDMcNoise) and isinstance(self.network, OpenAIWrapper)
                and isinstance(self.network.diffusion_model, VideoUNet) and "num_video_frames" in self.kwargs)


class _FusedState:
    """Per-(shape) fused step executor bound to one VideoUNet launch plan."""

    def __init__(self, unet: VideoUNet, F_: int, H: int, W: int, T: int, scale: torch.Tensor, shard=None):
        self.plan = unet.get_plan(2 * F_, H, W, T, shard=shard)
        dev = unet.device
        self.scale = scale.reshape(-1).to(device=dev, dtype=torch.float32).contiguous()
        self.key = None
        self.cc = self.cuc = None
        # CUDA-graph replay of the whole step (pre -> ~750 launches -> post): static I/O buffers + one graph.  Frame-sharded
        # plans are captured too when their exchanges are peer-memory kernels (every rank replays the same graph, the flag
        # barriers inside it keep the ranks in step); with NCCL exchanges the step stays eager.
        self.use_graph = os.environ.get("HI3D_CUDA_GRAPH", "1") != "0" and (shard is None or self.plan.exchange_mode == "peer")
        self._graph = None
        self._gx = torch.zeros(F_, 4, H, W, dtype=torch.float32, device=dev)
        self._gxo = torch.zeros_like(self._gx)
        self._gs = torch.ones(F_, dtype=torch.float32, device=dev)
        self._gsn = torch.ones(F_, dtype=torch.float32, device=dev)

    def set_conditioning(self, c: dict, uc: dict):
        ctx = torch.cat((uc["crossattn"], c["crossattn"]), 0)
        y = torch.cat((uc["vector"], c["vector"]), 0)
        self.plan.prepare_conditioning(ctx, y)
        cc, cuc = c.get("concat", None), uc.get("concat", None)
        if cc is None:
            if self.cc is not None:
                self._graph = None
            self.cc = self.cuc = None
            return
        dt = cc.dtype if cc.dtype in (torch.float16, torch.float32) else torch.float32
        if self.cc is None or self.cc.shape != cc.shape or self.cc.dtype != dt:
            # persistent copies: their addresses are baked into the captured graph
            self.cc, self.cuc = torch.empty_like(cc, dtype=dt).contiguous(), torch.empty_like(cc, dtype=dt).contiguous()
            self._graph = None
        self.cc.copy_(cc)
        if cuc is None:
            self.cuc.zero_()
        else:
            self.cuc.copy_(cuc)

    @staticmethod
    def cond_key(c: dict, uc: dict):
        return tuple((k, d[k].data_ptr(), d[k]._version, tuple(d[k].shape)) for d in (c, uc) for k in sorted(d)
                     if torch.is_tensor(d[k]))

    def _launch(self, x, sigma, next_sigma, x_out, den):
        plan = self.plan
        F_, Cx, H, W = x.shape
        ops.sampler_pre(x, sigma, self.cuc, self.cc, plan.xin.t.view(2 * F_, H, W, CIN_PAD), c_noise_out=plan.t_in)
        plan.run()
        ops.sampler_post(plan.net_out.t, x, sigma, next_sigma, self.scale, x_out, den)

    def denoise(self, x: torch.Tensor, sigma: torch.Tensor) -> torch.Tensor:
        """Guided denoised latents D(x, sigma) on the fused path (sampler_pre -> launch plan -> sampler_post): the network
        evaluation of ANY sampler (Heun's second evaluation, DPM-Solver++), without the Euler update."""
        plan = self.plan
        x = x.contiguous()
        sigma = sigma.contiguous()
        F_, Cx, H, W = x.shape
        ops.sampler_pre(x, sigma, self.cuc, self.cc, plan.xin.t.view(2 * F_, H, W, CIN_PAD), c_noise_out=plan.t_in)
        plan.run()
        den = torch.empty_like(x)
        if getattr(self, "_scratch", None) is None or self._scratch.shape != x.shape:
            self._scratch = torch.empty_like(x)
        ops.sampler_post(plan.net_out.t, x, sigma, sigma, self.scale, self._scratch, den)
        return den

    def step(self, x: torch.Tensor, sigma: torch.Tensor, next_sigma: torch.Tensor, want_denoised: bool = False):
        if self.use_graph and not want_denoised and x.shape == self._gx.shape:
            self._gx.copy_(x)
            self._gs.copy_(sigma)
            self._gsn.copy_(next_sigma)
            if self._graph is None:
                self._launch(self._gx, self._gs, self._gsn, self._gxo, None)        # eager warm-up (lazy one-time init)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = _native.launch_count()
                with torch.cuda.graph(g):
                    self._launch(self._gx, self._gs, self._gsn, self._gxo, None)
                self._graph_launches = _native.launch_count() - n0
                _native.note_graph_replay(-self._graph_launches)      # capture-time calls did not execute
                self._graph = g
            self._graph.replay()
            _native.note_graph_replay(self._graph_launches)
            return self._gxo.clone()
        plan = self.plan
        x = x.contiguous()
        sigma, next_sigma = sigma.contiguous(), next_sigma.contiguous()
        F_, Cx, H, W = x.shape
        ops.sampler_pre(x, sigma, self.cuc, self.cc, plan.xin.t.view(2 * F_, H, W, CIN_PAD), c_noise_out=plan.t_in)
        plan.run()
        x_out = torch.empty_like(x)
        den = torch.empty_like(x) if want_denoised else None
        ops.sampler_post(plan.net_out.t, x, sigma, next_sigma, self.scale, x_out, den)
        return (x_out, den) if want_denoised else x_out


# ------------------------------------------------------------------------------------------------------------
# samplers
# ------------------------------------------------------------------------------------------------------------
DEFAULT_GUIDER = {"target": "sgm.modules.diffusionmodules.guiders.IdentityGuider"}


class BaseDiffusionSampler:
    def __init__(self, discretization_config, num_steps: Union[int, None] = None, guider_config=None,
                 verbose: bool = False, device: str = "cuda"):
        self.num_steps = num_steps
        self.discretization = instantiate_from_config(discretization_config)
        self.guider = instantiate_from_config(default(guider_config, DEFAULT_GUIDER))
        self.verbose = verbose
        self.device = device
        self._fused: Dict[tuple, _FusedState] = {}

    def prepare_sampling_loop(self, x, cond, uc=None, num_steps=None):
        sigmas = self.discretization(self.num_steps if num_steps is None else num_steps, device=self.device)
        uc = default(uc, cond)
        x *= torch.sqrt(1.0 + sigmas[0] ** 2.0)
        num_sigmas = len(sigmas)
        s_in = x.new_ones([x.shape[0]])
        return x, s_in, sigmas, num_sigmas, cond, uc

    def denoise(self, x, denoiser, sigma, cond, uc):
        """sampling.py:54-57.  When `denoiser` is a fusable binding the guided D(x, sigma) comes from the fused kernels (one
        network evaluation = sampler_pre -> launch plan -> sampler_post), whatever the solver around it is."""
        st = self._fused_state(denoiser, x, cond, default(uc, cond), refresh=False)
        if st is not None:
            return st.denoise(x, sigma)
        if isinstance(denoiser, FusedDenoiser) and denoiser.shard is not None:
            raise NotImplementedError("frame-sharded sampling needs the fused path (LinearPredictionGuider + "
                                      f"VScalingWithEDMcNoise, fp32 CUDA latents); got {type(self.guider).__name__}, x {x.dtype}")
        denoised = denoiser(*self.guider.prepare_inputs(x, sigma, cond, uc))
        return self.guider(denoised, sigma)

    # -- fused path (shared by every sampler) -------------------------------------------------------------------
    def _fused_state(self, denoiser, x, cond, uc, refresh: bool) -> Optional[_FusedState]:
        if not (isinstance(denoiser, FusedDenoiser) and denoiser.fusable()
                and isinstance(self.guider, LinearPredictionGuider) and x.is_cuda and x.dtype == torch.float32):
            return None
        unet = denoiser.network.diffusion_model
        T = int(denoiser.kwargs["num_video_frames"])
        if T != self.guider.num_frames:
            return None
        shard = denoiser.shard
        scale = self.guider.scale.reshape(-1)
        if shard is not None:             # this rank holds frames [rank*Tl, (rank+1)*Tl) of every clip
            if T % shard[1]:
                raise ValueError(f"{T} frames cannot be sharded over {shard[1]} ranks")
            Tl = T // shard[1]
            scale = scale[shard[0] * Tl:(shard[0] + 1) * Tl]
            T = Tl
        if x.shape[0] % T:
            return None
        F_, _, H, W = x.shape
        pkey = unet.plan_key(2 * F_, H, W, T, shard)       # holds the engine and the deterministic-mode switch
        key = (id(unet),) + pkey
        st = self._fused.get(key)
        if st is None or st.plan is not unet._plans.get(pkey):
            st = self._fused[key] = _FusedState(unet, F_, H, W, T, scale, shard)
        ck = _FusedState.cond_key(cond, uc)
        if refresh or st.key != ck:
            st.set_conditioning(cond, uc)
            st.key = ck
        return st


    def get_sigma_gen(self, num_sigmas):
        sigma_generator = range(num_sigmas - 1)
        if self.verbose:
            try:
                from tqdm import tqdm
                sigma_generator = tqdm(sigma_generator, total=num_sigmas,
                                       desc=f"Sampling with {self.__class__.__name__} for {num_sigmas} steps")
            except ImportError:
                pass
        return sigma_generator


class SingleStepDiffusionSampler(BaseDiffusionSampler):
    def sampler_step(self, sigma, next_sigma, denoiser, x, cond, uc, *args, **kwargs):
        raise NotImplementedError

    def euler_step(self, x, d, dt):
        return x + dt * d


class EDMSampler(SingleStepDiffusionSampler):
    def __init__(self, s_churn=0.0, s_tmin=0.0, s_tmax=float("inf"), s_noise=1.0, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.s_churn, self.s_tmin, self.s_tmax, self.s_noise = s_churn, s_tmin, s_tmax, s_noise

    def _gamma(self, sigmas, i, num_sigmas):
        if self.s_churn == 0.0:       # avoids the reference's per-step D2H sync (sampling.py:112,134)
            return 0.0
        return min(self.s_churn / (num_sigmas - 1), 2 ** 0.5 - 1) if self.s_tmin <= sigmas[i] <= self.s_tmax else 0.0

    def possible_correction_step(self, euler_step, x, d, dt, next_sigma, denoiser, cond, uc):
        return euler_step

    def sampler_step(self, sigma, next_sigma, denoiser, x, cond, uc=None, gamma=0.0, _refresh=False):
        if gamma == 0:
            st = self._fused_state(denoiser, x, cond, default(uc, cond), _refresh)
            if st is not None and type(self).possible_correction_step is EDMSampler.possible_correction_step:
                return st.step(x, sigma, next_sigma)
        sigma_hat = sigma * (gamma + 1.0)
        if gamma > 0:
            eps = torch.randn_like(x) * self.s_noise
            x = x + eps * append_dims(sigma_hat ** 2 - sigma ** 2, x.ndim) ** 0.5
        denoised = self.denoise(x, denoiser, sigma_hat, cond, uc)
        d = (x - denoised) / append_dims(sigma_hat, x.ndim)            # to_d, sampling_utils.py:34
        dt = append_dims(next_sigma - sigma_hat, x.ndim)
        self._heun_ctx = (next_sigma - sigma_hat).float().contiguous() if x.is_cuda else None
        euler_step = self.euler_step(x, d, dt)
        return self.possible_correction_step(euler_step, x, d, dt, next_sigma, denoiser, cond, uc)

    def step_call(self, denoiser, x, i, s_in, sigmas, num_sigmas, cond, uc):
        """Hi3D addition (sampling.py:109-124): one externally driven step of the loop."""
        gamma = self._gamma(sigmas, i, num_sigmas)
        return self.sampler_step(s_in * sigmas[i], s_in * sigmas[i + 1], denoiser, x, cond, uc, gamma,
                                 _refresh=(i == 0))

    def __call__(self, denoiser, x, cond, uc=None, num_steps=None):
        x, s_in, sigmas, num_sigmas, cond, uc = self.prepare_sampling_loop(x, cond, uc, num_steps)
        for i in self.get_sigma_gen(num_sigmas):
            gamma = self._gamma(sigmas, i, num_sigmas)
            x = self.sampler_step(s_in * sigmas[i], s_in * sigmas[i + 1], denoiser, x, cond, uc, gamma,
                                  _refresh=(i == 0))
        return x


class EulerEDMSampler(EDMSampler):
    """sampling.py:228-232: EDMSampler whose correction step is the identity (inherited)."""


# ------------------------------------------------------------------------------------------------------------
# SURVEY §8(f) N4: the two other samplers of the sgm surface that Hi3D-style configs can name.  Every network evaluation goes
# through `self.denoise`, i.e. the fused sampler_pre -> launch plan -> sampler_post kernels when the denoiser binding is fusable
# (guider, Denoiser scalings and the OpenAIWrapper concat included); the solver algebra on the (F, 4, h, w) fp32 state is one
# hi3d_sampler_lincomb4 launch per update on CUDA (plain tensor expressions on CPU, where they are checked against the
# unmodified reference classes).
# ------------------------------------------------------------------------------------------------------------
class HeunEDMSampler(EDMSampler):
    """sampling.py:236-254.  Second order: the slope at (x, sigma_hat) is averaged with the slope at the Euler point
    (x_e, sigma_next); the last step (sigma_next = 0) stays first order, which also saves one evaluation."""

    def possible_correction_step(self, euler_step, x, d, dt, next_sigma, denoiser, cond, uc):
        if float(next_sigma.sum()) < 1e-14:
            return euler_step
        sig_n = append_dims(next_sigma, x.ndim)
        den_next = self.denoise(euler_step, denoiser, next_sigma, cond, uc)
        if x.is_cuda and x.dtype == torch.float32 and getattr(self, "_heun_ctx", None) is not None:
            # x + dt/2 (d + d'),  d' = (x_e - D')/sigma':  one hi3d_sampler_lincomb4 launch over (x, d, x_e, D')
            dtv = self._heun_ctx                                                  # dt per sample, fp32 [F]
            h = 0.5 * dtv
            one = torch.ones_like(dtv)
            return ops.sampler_lincomb(torch.empty_like(x), [(x.contiguous(), one), (d.contiguous(), h),
                                                             (euler_step.contiguous(), h / next_sigma),
                                                             (den_next.contiguous(), -h / next_sigma)])
        d_next = (euler_step - den_next) / sig_n
        heun = x + (d + d_next) / 2.0 * dt
        return torch.where(sig_n > 0.0, heun, euler_step)


class DPMPP2MSampler(BaseDiffusionSampler):
    """sampling.py:305-379 (DPM-Solver++(2M), Lu et al. 2022) in t = -log(sigma): one evaluation per step; from the
    second step on the denoised estimate is extrapolated with the previous one (ratio r of the two log-step sizes)."""

    @staticmethod
    def _t(sigma):                       # sampling_utils.py: to_neg_log_sigma
        return sigma.log().neg()

    @staticmethod
    def _sigma(t):                       # sampling_utils.py: to_sigma
        return t.neg().exp()

    def sampler_step(self, old_denoised, previous_sigma, sigma, next_sigma, denoiser, x, cond, uc=None):
        denoised = self.denoise(x, denoiser, sigma, cond, uc)
        t, t_next = self._t(sigma), self._t(next_sigma)
        h = t_next - t
        keep = append_dims(self._sigma(t_next) / self._sigma(t), x.ndim)     # sigma_next / sigma
        gain = append_dims((-h).expm1(), x.ndim)                             # exp(-h) - 1 <= 0
        fused = x.is_cuda and x.dtype == torch.float32
        if old_denoised is None or float(next_sigma.sum()) < 1e-14:
            if fused:        # (sigma'/sigma) x - expm1(-h) D : one hi3d_sampler_lincomb4 launch
                k1, g1 = (self._sigma(t_next) / self._sigma(t)).float().contiguous(), (-(-h).expm1()).float().contiguous()
                return ops.sampler_lincomb(torch.empty_like(x), [(x.contiguous(), k1), (denoised.contiguous(), g1)]), denoised
            return keep * x - gain * denoised, denoised
        r = (t - self._t(previous_sigma)) / h
        if fused:            # (sigma'/sigma) x - expm1(-h) ((1 + 1/(2r)) D - 1/(2r) D_old)
            k1, g1 = (self._sigma(t_next) / self._sigma(t)).float().contiguous(), (-(-h).expm1()).float()
            return ops.sampler_lincomb(torch.empty_like(x), [(x.contiguous(), k1),
                                                             (denoised.contiguous(), (g1 * (1 + 1 / (2 * r))).contiguous()),
                                                             (old_denoised.contiguous(), (-g1 / (2 * r)).contiguous())]), denoised
        x_first = keep * x - gain * denoised
        w_new, w_old = append_dims(1 + 1 / (2 * r), x.ndim), append_dims(1 / (2 * r), x.ndim)
        x_second = keep * x - gain * (w_new * denoised - w_old * old_denoised)
        return torch.where(append_dims(next_sigma, x.ndim) > 0.0, x_second, x_first), denoised

    def __call__(self, denoiser, x, cond, uc=None, num_steps=None, **kwargs):
        x, s_in, sigmas, num_sigmas, cond, uc = self.prepare_sampling_loop(x, cond, uc, num_steps)
        prev_d = None
        for i in self.get_sigma_gen(num_sigmas):
            x, prev_d = self.sampler_step(prev_d, None if i == 0 else s_in * sigmas[i - 1], s_in * sigmas[i],
                                          s_in * sigmas[i + 1], denoiser, x, cond, uc=uc)
        return x
