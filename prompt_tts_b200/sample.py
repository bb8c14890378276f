"""Diffusion sampling on the B200 path (SURVEY section 8 row N1 -- not in the reference tree, which ships no sampler).

The loop is what a user of the reference would write with diffusers 0.15 on top of `TTSSingleSpeaker`:

    scheduler = DDPMScheduler(num_train_timesteps=1000)           # train.py:32-36 (linear betas 1e-4 .. 0.02, epsilon prediction)
    scheduler.set_timesteps(100)
    text_emb = model.text_encoder(ids, mask)                      # once
    for t in scheduler.timesteps:                                 # 990, 980, ..., 0
        eps = model.unet(x, t, encoder_hidden_states=text_emb).sample
        x = scheduler.step(eps, t, x).prev_sample

Here the text encoder runs once, the cross-attention K/V projections of its output are computed once and reused by all
steps (they do not depend on x or t), one denoiser forward is captured in a CUDA graph and replayed per step, and the
scheduler step is one fused kernel (`pt_ddpm_step`), optionally in-painting the first `prompt` frames from a noised copy
of the speech prompt (the builder-defined prompt protocol of SURVEY 8d config 4).

`DDIMSampler` and `DPMSolverSampler` run the same loop with diffusers 0.15's `DDIMScheduler` (default 50 steps) and
`DPMSolverMultistepScheduler` (DPM-Solver++ order 2, default 20 steps) on the same trained model: one denoiser forward per step,
so the cost of a sample is proportional to the step count.  Their steps are `pt_ddim_step` / `pt_dpmpp_step`, which in-paint the
prompt frames inside the kernel.

Classifier-free guidance (`sample(..., guidance_scale=w)`, all three samplers) follows diffusers 0.15's pipelines: with w > 1 each
step runs the denoiser once at batch 2B -- rows [0, B) conditioned on the text, rows [B, 2B) on the null condition (an all-zero
context, what condition dropout trains: `DenoiserTrainStep(..., cond_keep=)`) -- and the step uses
eps = eps_u + w (eps_c - eps_u) (`pt_cfg_combine`).  The null rows' cross-attention is exactly to_out's bias added to the residual
(ldm/attention.py:BasicTransformerBlock._cross_guided), so it is computed as that.  w = 1 (the default) is the unguided loop.

Prediction type (all three samplers, keyword `prediction_type`, as diffusers' schedulers take it): the model output is eps
("epsilon", the default, the reference's), x0 ("sample") or v ("v_prediction"), matching what the model was trained to predict
(`DenoiserTrainStep(..., prediction_type=)`).  Every type calls the `_pred` step entry points with the type; they convert the output
as diffusers 0.15's `step` does inside the same single pass.  Guidance combines the raw outputs whatever they parameterise, as
diffusers' pipelines do.
"""
from __future__ import annotations

import math
import numbers
from typing import Dict, List, Optional

import numpy as np
import torch

from . import engine as E
from . import ops


def ddpm_alphas_cumprod(n: int = 1000, beta_start: float = 1e-4, beta_end: float = 0.02) -> torch.Tensor:
    betas = torch.linspace(beta_start, beta_end, n, dtype=torch.float32)
    return torch.cumprod(1.0 - betas, 0)


def _check_guidance(name: str, w) -> float:
    if isinstance(w, bool) or not isinstance(w, numbers.Real) or not math.isfinite(float(w)) or float(w) < 1.0:
        raise ValueError(f"{name}: guidance_scale must be a finite real number >= 1 (1 = no guidance), got {w!r}")
    return float(w)


class _Sampler:
    """The sampling loop every scheduler shares: text encoder once, cross-attention K/V cached, one denoiser forward captured at
    call 1 and replayed; `_step` is the scheduler's update of x in place from the eps the forward left in `_static["eps"]`."""
    timesteps: List[int]

    def __init__(self, model, n_infer: int, use_graph: bool, prediction_type: str):
        self.pred_type, _ = ops.check_prediction(type(self).__name__, prediction_type)
        self.prediction_type = prediction_type
        self.model = model
        self.n_infer = n_infer
        self.acp = ddpm_alphas_cumprod()                      # host copy: the step coefficients are scalars per step
        self.use_graph = use_graph
        self.cache = E.get_cache(model)
        self._graph = None
        self._static: Dict[str, torch.Tensor] = {}

    # ---- one denoiser forward on static buffers (x, t) -> eps, with the text encoding and its K/V projections held fixed.
    # Guided: x2 = [x | copy of x] at batch 2B, the second half with the null condition, eps = the guided combination of the halves.
    def _denoise(self) -> None:
        tape = E.Tape(self.cache, recording=False)
        tape.kv_cache = self._kv
        x2 = self._static.get("x2")
        if x2 is None:
            y, _ = self.model.unet._fwd(tape, self._static["x"], self._static["t"], self._enc)
            self._static["eps"].copy_(y)
            return
        B = x2.shape[0] // 2
        x2[B:].copy_(x2[:B])
        tape.cond_rows = B
        y, _ = self.model.unet._fwd(tape, x2, self._static["t"], self._enc)
        eps = self._static["eps"]
        ops.call("cfg_combine", ops._p(y), ops._p(eps), eps.numel(), self._w, ops._stream())

    def _start(self, x: torch.Tensor, prompt: Optional[torch.Tensor], prompt_noise: Optional[torch.Tensor], keep: int) -> None:
        """per-call state of the scheduler step"""
        raise NotImplementedError

    def _step(self, i: int, t: int, x: torch.Tensor, noises: Optional[torch.Tensor], gen: torch.Generator) -> None:
        raise NotImplementedError

    def _step_call(self, name: str, *args) -> None:
        """the scheduler's step kernel `pt_<name>_pred` for the model's prediction type"""
        ops.call(name + "_pred", *args, self.pred_type, ops._stream())

    def _draw_noise(self, i: int, noises: Optional[torch.Tensor], gen: torch.Generator) -> None:
        """the step's noise buffer: noises[i] when given, else a draw from the sampler's generator"""
        if noises is not None:
            self._noise.copy_(noises[i])
        else:
            self._noise.normal_(generator=gen)

    @torch.no_grad()
    def sample(self, ids: torch.Tensor, T: int, x_T: Optional[torch.Tensor] = None, noises: Optional[torch.Tensor] = None,
               prompt: Optional[torch.Tensor] = None, prompt_noise: Optional[torch.Tensor] = None, seed: int = 0,
               return_codes: bool = False, prompt_tokens: Optional[torch.Tensor] = None, guidance_scale: float = 1.0) -> torch.Tensor:
        """ids int32 [B, Lt]; returns x_0 fp32 [B, C, T] (or int64 codes in [0, 1023] with return_codes).
        x_T / noises[n_infer, B, C, T] / prompt_noise may be given for reproducibility against an oracle; otherwise they are
        drawn from a generator seeded with `seed` (noises is read only at the steps that add noise).  prompt fp32 [B, C, P]:
        clean prompt frames in-painted at every step, noised to the level the step lands on (clean at the last step).
        prompt_tokens float [B, P, cross_attention_dim] (optional, default off): a speech-prompt encoding appended to the text
        encoding as extra cross-attention tokens -- `Unet1DConditionModel.forward` takes `encoder_hidden_states` of any length
        (unet_1d_condition.py:557); with None the conditioning is exactly the reference's.
        guidance_scale w >= 1: classifier-free guidance for w > 1 (module docstring); x_T, noises, the prompt and prompt tokens act
        on the B guided rows exactly as without guidance.  The model should have been trained with condition dropout."""
        w = _check_guidance(type(self).__name__, guidance_scale)
        if not ids.is_cuda:
            raise ops._lib.PtError(f"{type(self).__name__}: inputs must be CUDA tensors; there is no CPU fallback")
        dev = ids.device
        B = ids.shape[0]
        Cin = self.model.unet.conv_in.weight.shape[1]
        gen = torch.Generator(device=dev).manual_seed(seed)
        x = x_T.clone().float() if x_T is not None else torch.randn(B, Cin, T, device=dev, generator=gen)
        guided = w > 1.0
        x2 = None
        if guided:      # the sampler's x is the first half of the 2B-row denoiser input: the step kernels update it in place
            x2 = torch.empty(2 * B, Cin, T, device=dev)
            x2[:B].copy_(x)
            x = x2[:B]
        self._w = w
        # text encoder once; K/V of every cross-attention layer are filled in by the first denoiser call and then reused
        tape = E.Tape(self.cache, recording=False)
        self._enc = self.model.text_encoder._fwd(tape, ids.to(torch.int32).contiguous())
        if prompt_tokens is not None:
            if prompt_tokens.shape[0] != B or prompt_tokens.shape[2] != self._enc.data.shape[2]:
                raise ops._lib.PtError(f"prompt_tokens must be [B, P, {self._enc.data.shape[2]}], got {tuple(prompt_tokens.shape)}")
            self._enc = E.Var(torch.cat([self._enc.data, ops.cast_bf16(prompt_tokens.float().contiguous())], dim=1), needs_grad=False)
        self._kv: Dict[int, E.Var] = {}
        self._static = {"x": x, "t": torch.zeros(2 * B if guided else B, dtype=torch.int64, device=dev), "eps": torch.empty_like(x)}
        if guided:
            self._static["x2"] = x2
        self._graph = None
        keep = 0
        if prompt is not None:
            keep = prompt.shape[-1]
            if prompt_noise is None:
                prompt_noise = torch.randn(self.n_infer, B, Cin, keep, device=dev, generator=gen)
        self._T = T
        self._start(x, prompt, prompt_noise, keep)
        for i, t in enumerate(self.timesteps):
            self._static["t"].fill_(t)
            if self.use_graph and i == 1:        # call 0 ran eagerly (fills the K/V cache, warms the weight packs); capture call 1
                torch.cuda.synchronize()
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._denoise()
                self._graph.replay()             # capture only records; this executes step 1
            elif self._graph is not None:
                self._graph.replay()
            else:
                self._denoise()
            self._step(i, t, x, noises, gen)
        self._graph = None
        if return_codes:
            codes = torch.empty(x.shape, dtype=torch.int64, device=dev)
            ops.call("codes_affine_inv", ops._p(x), ops._p(codes), x.numel(), ops._stream())
            return codes
        return x.clone() if guided else x      # guided: not a view that keeps the 2B-row buffer alive


class DDPMSampler(_Sampler):
    def __init__(self, model, n_infer: int = 100, n_train: int = 1000, use_graph: bool = True, *, prediction_type: str = "epsilon"):
        n_infer = _check_steps("DDPMSampler", n_infer, n_train)
        super().__init__(model, n_infer, use_graph, prediction_type)
        self.n_train = n_train
        self.stride = n_train // n_infer
        self.acp = ddpm_alphas_cumprod(n_train)
        self.timesteps = [i * self.stride for i in range(n_infer)][::-1]

    def _start(self, x, prompt, prompt_noise, keep):
        self._prompt, self._prompt_noise, self._keep = prompt, prompt_noise, keep
        self._known = torch.zeros_like(x) if prompt is not None else None
        self._noise = torch.empty_like(x)

    def _step(self, i, t, x, noises, gen):
        known, noise, keep = self._known, self._noise, self._keep
        t_prev = t - self.stride
        acp_t = float(self.acp[t])
        acp_prev = float(self.acp[t_prev]) if t_prev >= 0 else 1.0
        if t_prev >= 0:
            self._draw_noise(i, noises, gen)
        if known is not None:
            # in-paint: the prompt frames of x_{t_prev} are the clean prompt noised to level t_prev (clean at the last step)
            sa, sb = (acp_prev ** 0.5, (1.0 - acp_prev) ** 0.5) if t_prev >= 0 else (1.0, 0.0)
            known[..., :keep] = sa * self._prompt + sb * self._prompt_noise[i]
        self._step_call("ddpm_step", ops._p(self._static["eps"]), ops._p(x), ops._p(noise if t_prev >= 0 else None), ops._p(known),
                        ops._p(x), x.numel(), self._T, keep, acp_t, acp_prev)


def _check_steps(name: str, n_infer, hi: int) -> int:
    if isinstance(n_infer, bool) or int(n_infer) != n_infer or not 1 <= int(n_infer) <= hi:
        raise ValueError(f"{name}: n_infer must be an integer in [1, {hi}], got {n_infer!r}")
    return int(n_infer)


class _KernelPromptSampler(_Sampler):
    """Samplers whose step kernel in-paints the prompt frames itself, from [B, C, P] and [n_infer, B, C, P] fp32 device buffers."""

    def _start_prompt(self, x, prompt, prompt_noise, keep):
        self._keep, self._prompt, self._prompt_noise = keep, None, None
        if prompt is None:
            return
        B, C, T = x.shape
        want = (self.n_infer, B, C, keep)
        if tuple(prompt.shape) != want[1:] or tuple(prompt_noise.shape) != want or keep > T or not (prompt.is_cuda and prompt_noise.is_cuda):
            raise ops._lib.PtError(f"{type(self).__name__}: prompt must be a CUDA tensor [B, C, P] = {want[1:]} with P <= T = {T} and "
                                   f"prompt_noise [n_infer, B, C, P] = {want}; got {tuple(prompt.shape)} / {tuple(prompt_noise.shape)}")
        self._prompt = prompt.float().contiguous()
        self._prompt_noise = prompt_noise.float().contiguous()

    def _prompt_args(self, i: int, acp_to: Optional[float]):
        """pointer / scale arguments of the in-kernel in-painting: the prompt noised to alphas_cumprod `acp_to`, clean for None"""
        if self._prompt is None:
            return ops._p(None), ops._p(None), 1.0, 0.0
        if acp_to is None:
            return ops._p(self._prompt), ops._p(None), 1.0, 0.0
        a = torch.tensor(acp_to, dtype=torch.float32)
        return ops._p(self._prompt), ops._p(self._prompt_noise[i]), float(torch.sqrt(a)), float(torch.sqrt(1 - a))


class DDIMSampler(_KernelPromptSampler):
    """diffusers 0.15 `DDIMScheduler` (clip_sample, set_alpha_to_one, steps_offset 0) over the training schedule: timesteps
    (n_infer - 1) * r, ..., r, 0 with r = 1000 // n_infer.  eta = 0 is deterministic; eta = 1 adds the DDPM posterior's noise."""

    def __init__(self, model, n_infer: int = 50, eta: float = 0.0, use_graph: bool = True, *, prediction_type: str = "epsilon"):
        n_infer = _check_steps("DDIMSampler", n_infer, 1000)
        if not 0.0 <= eta <= 1.0:
            raise ValueError(f"DDIMSampler: eta must be in [0, 1] (DDIM's interpolation between deterministic and DDPM noise), got {eta!r}")
        super().__init__(model, n_infer, use_graph, prediction_type)
        self.eta = float(eta)
        self.stride = 1000 // n_infer
        self.timesteps = [i * self.stride for i in range(n_infer)][::-1]

    def _start(self, x, prompt, prompt_noise, keep):
        self._start_prompt(x, prompt, prompt_noise, keep)
        self._noise = torch.empty_like(x) if self.eta > 0 else None

    def _step(self, i, t, x, noises, gen):
        t_prev = t - self.stride
        acp_prev = float(self.acp[t_prev]) if t_prev >= 0 else 1.0
        if self._noise is not None:
            self._draw_noise(i, noises, gen)
        pp, pn, pa, pb = self._prompt_args(i, acp_prev if t_prev >= 0 else None)
        self._step_call("ddim_step", ops._p(self._static["eps"]), ops._p(x), ops._p(self._noise), pp, pn, ops._p(x), x.numel(), x.shape[-1],
                        self._keep, float(self.acp[t]), acp_prev, self.eta, pa, pb)


class DPMSolverSampler(_KernelPromptSampler):
    """diffusers 0.15 `DPMSolverMultistepScheduler` (DPM-Solver++, order 2, midpoint, lower_order_final): timesteps
    round(linspace(0, 999, n_infer + 1))[::-1][:-1]; the last step lands at t = 0.  First order at the first step (and at the
    last one when n_infer < 15), second order from the x0 prediction of the previous step otherwise.  n_infer <= 999: at 1000 the
    rounded grid repeats a timestep."""

    def __init__(self, model, n_infer: int = 20, use_graph: bool = True, *, prediction_type: str = "epsilon"):
        n_infer = _check_steps("DPMSolverSampler", n_infer, 999)
        super().__init__(model, n_infer, use_graph, prediction_type)
        self.timesteps = np.linspace(0, 999, n_infer + 1).round()[::-1][:-1].astype(np.int64).tolist()

    def _start(self, x, prompt, prompt_noise, keep):
        self._start_prompt(x, prompt, prompt_noise, keep)
        self._m = torch.empty_like(x)            # x0 prediction of the previous step, overwritten with this step's in the kernel

    def _step(self, i, t, x, noises, gen):
        n = self.n_infer
        last = i == n - 1
        t_to = 0 if last else self.timesteps[i + 1]
        order = 1 if i == 0 or (last and n < 15) else 2
        acp_s1 = float(self.acp[self.timesteps[i - 1]]) if order == 2 else 0.0
        pp, pn, pa, pb = self._prompt_args(i, None if last else float(self.acp[t_to]))
        self._step_call("dpmpp_step", ops._p(self._static["eps"]), ops._p(x), ops._p(self._m), ops._p(self._m), pp, pn, ops._p(x), x.numel(),
                        x.shape[-1], self._keep, float(self.acp[t]), acp_s1, float(self.acp[t_to]), order, pa, pb)
