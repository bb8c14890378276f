"""The reference's training step (train.py:86-120) on the B200 path, without the autograd bridge:

    noise ~ N(0,1); t ~ U{0..999}; x_t = sqrt(acp_t) x0 + sqrt(1-acp_t) noise      (DDPMScheduler.add_noise, :96-98)
    pred = model(x_t, t, ids, mask).sample                                          (:100-105)
    loss = mse(pred, noise); loss.backward()                                        (:107,115)

`DenoiserTrainStep` runs add_noise -> tape forward -> MSE (+ its gradient) -> tape backward with static buffers so the
whole step can be captured in one CUDA graph; parameter gradients land in `param.grad` (fp32 views of one flat buffer with
the reference's logical shapes), so the reference's `clip_grad_norm_` / `AdamW` lines keep working on top of it.  As with
`zero_grad()` after every optimiser step in the reference (train.py:120), each accumulation window starts from zero.

Classifier-free guidance training (not in the reference tree): `cond_keep` (bool [B]) replaces the text encoding of the samples
where it is False with the null condition, an all-zero context, before the denoiser sees it (condition dropout).  The caller draws
the mask each step, e.g. `torch.rand(B, device=dev) >= p_uncond`, as it draws `noise` and `t`.

Prediction type and Min-SNR weighting (not in the reference tree, which trains epsilon prediction): with
`DenoiserTrainStep(..., prediction_type="v_prediction" | "sample")` the loss target is diffusers' `get_velocity(x0, noise, t)` or
x0 instead of `noise`, and `snr_gamma=g` weights each sample's MSE by Min-SNR-g (`compute_snr` of diffusers' training examples:
min(snr, g) / snr for epsilon, / (snr + 1) for v, min(snr, g) for sample).  The target and the weight are formed inside one kernel
(`pt_diffusion_loss`), from `t` on the device.  The samplers must be built with the same `prediction_type`.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import engine as E
from . import ops
from .sample import ddpm_alphas_cumprod


def ddpm_tables(n: int = 1000, beta_start: float = 1e-4, beta_end: float = 0.02, device="cuda"):
    """sqrt(alphas_cumprod), sqrt(1 - alphas_cumprod) of the linear-beta DDPM schedule (train.py:32-36)."""
    acp = ddpm_alphas_cumprod(n, beta_start, beta_end)
    return (acp ** 0.5).to(device), ((1 - acp) ** 0.5).to(device)


class DenoiserTrainStep:
    def __init__(self, model, grad_sync=None, accumulation_steps: int = 1, *, prediction_type: str = "epsilon",
                 snr_gamma: Optional[float] = None):
        """grad_sync: a `prompt_tts_b200.dp.GradSync` (flat gradient buffer; overlaps the gradient all-reduce with the backward
        sweep when world_size > 1); built for a single process when omitted.
        accumulation_steps: the reference's `gradient_accumulation_steps` (train.py:27,80 `accelerator.accumulate`): every call is
        one micro-step; the flat gradient buffer is cleared at the first micro-step of a window, the loss gradient is scaled by
        1 / accumulation_steps (what `accelerator.backward` does), ranks exchange gradients only during the last micro-step, and
        `sync_gradients` tells the optimiser wrapper whether to step (`FusedClipAdamW.step` is a no-op otherwise).
        prediction_type: "epsilon" (the reference's), "sample" or "v_prediction" -- diffusers' scheduler option of that name.
        snr_gamma: None (unweighted, the reference's) or gamma > 0 of Min-SNR-gamma loss weighting (module docstring)."""
        self.pred_type, self._snr_gamma = ops.check_prediction("DenoiserTrainStep", prediction_type, snr_gamma)
        self.prediction_type = prediction_type
        self.model = model
        self.params = [p for p in model.parameters()]
        self.cache = E.get_cache(model)
        self.sa: Optional[torch.Tensor] = None
        self.sb: Optional[torch.Tensor] = None
        if grad_sync is None:      # single GPU: still use the flat gradient buffer (one memset per step, no per-tensor zero fills)
            from .dp import GradSync
            grad_sync = GradSync(model, world_size=1)
        self.grad_sync = grad_sync
        self.accumulation_steps = max(1, int(accumulation_steps))
        self.micro = 0
        self.sync_gradients = True
        self.loss = None

    @staticmethod
    def _check(x0, noise, t, ids):
        """The kernels read raw pointers: an int64 `ids` would be read as alternating low words and zeros, an int32 `t` would
        index the schedule tables out of bounds.  nn.Embedding / the scheduler accept either, so convert here."""
        if not (x0.is_cuda and noise.is_cuda and t.is_cuda and ids.is_cuda):
            raise ops._lib.PtError("DenoiserTrainStep: inputs must be CUDA tensors; there is no CPU fallback")
        if x0.shape != noise.shape or x0.dim() != 3:
            raise ops._lib.PtError(f"DenoiserTrainStep: x0 {tuple(x0.shape)} and noise {tuple(noise.shape)} must both be [B, C, T]")
        if t.shape != (x0.shape[0],) or ids.dim() != 2 or ids.shape[0] != x0.shape[0]:
            raise ops._lib.PtError(f"DenoiserTrainStep: t {tuple(t.shape)} must be [B] and ids {tuple(ids.shape)} [B, Lt]")
        if x0.dtype != torch.float32 or not x0.is_contiguous():
            x0 = x0.float().contiguous()
        if noise.dtype != torch.float32 or not noise.is_contiguous():
            noise = noise.float().contiguous()
        if t.dtype != torch.int64 or not t.is_contiguous():
            t = t.to(torch.int64).contiguous()
        if ids.dtype != torch.int32 or not ids.is_contiguous():
            ids = ids.to(torch.int32).contiguous()
        return x0, noise, t, ids

    def __call__(self, x0, noise, t, ids, mask=None, loss_out: Optional[torch.Tensor] = None, gscale: float = 1.0,
                 cond_keep: Optional[torch.Tensor] = None):
        """x0, noise fp32 [B, C, T]; t int64 [B] in [0, 1000); ids int32 [B, Lt] (other integer / float dtypes are converted).
        cond_keep: optional bool / uint8 [B] on the same device, 0 = train this sample unconditionally (all-zero text context);
        read from device memory, so a captured step replays with whatever mask was last written into the same buffer.
        Returns the loss of this micro-batch (0-d fp32 CUDA tensor)."""
        x0, noise, t, ids = self._check(x0, noise, t, ids)
        keep = E.cond_keep_mask(cond_keep, x0.shape[0], x0.device, "DenoiserTrainStep") if cond_keep is not None else None
        if self.sa is None:
            self.sa, self.sb = ddpm_tables(device=x0.device)
        first = self.micro == 0
        last = self.micro == self.accumulation_steps - 1
        self.sync_gradients = last
        self.micro = 0 if last else self.micro + 1
        B = x0.shape[0]
        xt = torch.empty_like(x0)
        ops.call("add_noise", ops._p(x0), ops._p(noise), ops._p(t), ops._p(self.sa), ops._p(self.sb), ops._p(xt), B, x0[0].numel(), ops._stream())
        tape = E.Tape(self.cache, recording=True)
        self.grad_sync.attach(tape, zero=first, sync=last)
        enc = self.model.text_encoder._fwd(tape, ids)
        if keep is not None:
            enc = E.cond_select(tape, enc, keep)
        pred, seed = self.model.unet._fwd(tape, xt, t, enc)
        loss = torch.zeros((), dtype=torch.float32, device=x0.device) if loss_out is None else loss_out.zero_()
        dpred = torch.empty_like(pred)
        gs = gscale / self.accumulation_steps
        if self.pred_type == 0 and self._snr_gamma == 0.0:
            ops.call("mse_fwd_bwd", ops._p(pred), ops._p(noise), ops._p(loss), ops._p(dpred), pred.numel(), gs, ops._stream())
        else:
            ops.call("diffusion_loss", ops._p(pred), ops._p(x0), ops._p(noise), ops._p(t), ops._p(self.sa), ops._p(self.sb), ops._p(loss),
                     ops._p(dpred), B, x0[0].numel(), self.pred_type, self._snr_gamma, gs, ops._stream())
        seed([dpred])
        tape.backward()
        self.grad_sync.finish()
        for p in self.params:
            g = tape.pgrads.get(id(p))
            if g is None:
                continue
            if p.grad is None or p.grad.data_ptr() != g.data_ptr():
                p.grad = g            # a view of the flat buffer (permuted for k=3 conv weights): holds the window's accumulated sum
        self.loss = loss
        return loss
