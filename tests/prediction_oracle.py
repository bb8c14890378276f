"""The oracle for sample / v prediction and Min-SNR-gamma weighting, restated from diffusers, on top of the oracle shim.

The shim's schedulers (oracle/diffusers_shim) restate epsilon prediction only.  The subclasses here add the "sample" and
"v_prediction" branches of diffusers 0.15's `DDPMScheduler.step` / `get_velocity`, `DDIMScheduler.step` and
`DPMSolverMultistepScheduler.convert_model_output`, restated from the published 0.15 code; their epsilon paths are the shim's.
`compute_snr` is restated from diffusers' training examples (`examples/text_to_image/train_text_to_image.py`, `--snr_gamma`): it
is not part of the 0.15 library.  Like the shim, parity with the real library is unpinned (no golden vectors from diffusers exist
offline).  `train_step_loss` and `ddpm_step` extend oracle/ref_model.py's functions of those names with a prediction type.
"""
import os
import sys

import torch
import torch.nn.functional as F

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(_ROOT, "oracle"))
sys.path.insert(0, os.path.join(_ROOT, "oracle", "diffusers_shim"))
import ref_model  # noqa: E402
from diffusers import DDPMScheduler as _DDPM  # noqa: E402
from diffusers.schedulers_few_step import DDIMScheduler as _DDIM  # noqa: E402
from diffusers.schedulers_few_step import DPMSolverMultistepScheduler as _DPM  # noqa: E402
from diffusers.schedulers_few_step import SchedulerOutput  # noqa: E402

PREDICTION_TYPES = ("epsilon", "sample", "v_prediction")


def _with_prediction_type(base, self, prediction_type, kw):
    """the shim's constructor (which takes epsilon only), then the configured prediction type"""
    if prediction_type not in PREDICTION_TYPES:
        raise ValueError(f"prediction_type given as {prediction_type} must be one of {PREDICTION_TYPES}")
    base.__init__(self, prediction_type="epsilon", **kw)
    self.config["prediction_type"] = prediction_type


class DDPMScheduler(_DDPM):
    """diffusers 0.15 DDPMScheduler (linear betas, fixed_small variance) with all three prediction types and `get_velocity`."""

    def __init__(self, prediction_type="epsilon", **kw):
        _with_prediction_type(_DDPM, self, prediction_type, kw)

    def get_velocity(self, sample, noise, timesteps):
        alphas_cumprod = self.alphas_cumprod.to(device=sample.device, dtype=sample.dtype)
        timesteps = timesteps.to(sample.device)
        sqrt_alpha_prod = (alphas_cumprod[timesteps] ** 0.5).flatten()
        while len(sqrt_alpha_prod.shape) < len(sample.shape):
            sqrt_alpha_prod = sqrt_alpha_prod.unsqueeze(-1)
        sqrt_one_minus_alpha_prod = ((1 - alphas_cumprod[timesteps]) ** 0.5).flatten()
        while len(sqrt_one_minus_alpha_prod.shape) < len(sample.shape):
            sqrt_one_minus_alpha_prod = sqrt_one_minus_alpha_prod.unsqueeze(-1)
        return sqrt_alpha_prod * noise - sqrt_one_minus_alpha_prod * sample

    def step(self, model_output, timestep, sample, generator=None, noise=None):
        if self.config.prediction_type == "epsilon":
            return super().step(model_output, timestep, sample, generator=generator, noise=noise)
        t = int(timestep)
        n = self.num_inference_steps if self.num_inference_steps else self.config.num_train_timesteps
        prev_t = t - self.config.num_train_timesteps // n
        a_t = self.alphas_cumprod[t]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.one
        b_t = 1 - a_t
        b_prev = 1 - a_prev
        cur_alpha = a_t / a_prev
        cur_beta = 1 - cur_alpha
        if self.config.prediction_type == "sample":
            x0 = model_output
        else:
            x0 = (a_t ** 0.5) * sample - (b_t ** 0.5) * model_output
        if self.config.clip_sample:
            x0 = x0.clamp(-1, 1)
        c0 = (a_prev ** 0.5 * cur_beta) / b_t
        ct = cur_alpha ** 0.5 * b_prev / b_t
        mean = c0 * x0 + ct * sample
        if t > 0:
            var = torch.clamp(b_prev / b_t * cur_beta, min=1e-20)
            if noise is None:
                noise = torch.randn(model_output.shape, generator=generator, dtype=model_output.dtype, device=model_output.device)
            mean = mean + var ** 0.5 * noise
        return mean


class DDIMScheduler(_DDIM):
    """diffusers 0.15 DDIMScheduler with all three prediction types.  For sample and v, eps is formed from the unclipped x0
    prediction, before `clip_sample` clamps it."""

    def __init__(self, prediction_type="epsilon", **kw):
        _with_prediction_type(_DDIM, self, prediction_type, kw)

    def step(self, model_output, timestep, sample, eta=0.0, use_clipped_model_output=False, generator=None,
             variance_noise=None, return_dict=True):
        if self.config.prediction_type == "epsilon":
            return super().step(model_output, timestep, sample, eta=eta, use_clipped_model_output=use_clipped_model_output,
                                generator=generator, variance_noise=variance_noise, return_dict=return_dict)
        timestep = int(timestep)
        prev_timestep = timestep - self.config.num_train_timesteps // self.num_inference_steps
        alpha_prod_t = self.alphas_cumprod[timestep]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        beta_prod_t = 1 - alpha_prod_t
        if self.config.prediction_type == "sample":
            pred_original_sample = model_output
            pred_epsilon = (sample - alpha_prod_t ** 0.5 * pred_original_sample) / beta_prod_t ** 0.5
        else:
            pred_original_sample = (alpha_prod_t ** 0.5) * sample - (beta_prod_t ** 0.5) * model_output
            pred_epsilon = (alpha_prod_t ** 0.5) * model_output + (beta_prod_t ** 0.5) * sample
        if self.config.clip_sample:
            pred_original_sample = pred_original_sample.clamp(-1, 1)
        variance = self._get_variance(timestep, prev_timestep)
        std_dev_t = eta * variance ** 0.5
        if use_clipped_model_output:
            pred_epsilon = (sample - alpha_prod_t ** 0.5 * pred_original_sample) / beta_prod_t ** 0.5
        pred_sample_direction = (1 - alpha_prod_t_prev - std_dev_t ** 2) ** 0.5 * pred_epsilon
        prev_sample = alpha_prod_t_prev ** 0.5 * pred_original_sample + pred_sample_direction
        if eta > 0:
            if variance_noise is None:
                variance_noise = torch.randn(model_output.shape, generator=generator, dtype=model_output.dtype,
                                             device=model_output.device)
            prev_sample = prev_sample + std_dev_t * variance_noise
        if not return_dict:
            return (prev_sample,)
        return SchedulerOutput(prev_sample, pred_original_sample)


class DPMSolverMultistepScheduler(_DPM):
    """diffusers 0.15 DPMSolverMultistepScheduler ("dpmsolver++", midpoint) with all three prediction types: the history holds the
    x0 prediction whatever the model parameterises."""

    def __init__(self, prediction_type="epsilon", **kw):
        _with_prediction_type(_DPM, self, prediction_type, kw)

    def convert_model_output(self, model_output, timestep, sample):
        if self.config.prediction_type == "epsilon":
            return super().convert_model_output(model_output, timestep, sample)
        if self.config.prediction_type == "sample":
            return model_output
        alpha_t, sigma_t = self.alpha_t[timestep], self.sigma_t[timestep]
        return alpha_t * sample - sigma_t * model_output


def compute_snr(noise_scheduler, timesteps):
    """Signal-to-noise ratio (alpha_t / sigma_t)^2 of `timesteps`, for Min-SNR-gamma loss weighting (Hang et al. 2023), as
    diffusers' training examples compute it."""
    alphas_cumprod = noise_scheduler.alphas_cumprod
    sqrt_alphas_cumprod = alphas_cumprod ** 0.5
    sqrt_one_minus_alphas_cumprod = (1.0 - alphas_cumprod) ** 0.5

    sqrt_alphas_cumprod = sqrt_alphas_cumprod.to(device=timesteps.device)[timesteps].float()
    while len(sqrt_alphas_cumprod.shape) < len(timesteps.shape):
        sqrt_alphas_cumprod = sqrt_alphas_cumprod[..., None]
    alpha = sqrt_alphas_cumprod.expand(timesteps.shape)

    sqrt_one_minus_alphas_cumprod = sqrt_one_minus_alphas_cumprod.to(device=timesteps.device)[timesteps].float()
    while len(sqrt_one_minus_alphas_cumprod.shape) < len(timesteps.shape):
        sqrt_one_minus_alphas_cumprod = sqrt_one_minus_alphas_cumprod[..., None]
    sigma = sqrt_one_minus_alphas_cumprod.expand(timesteps.shape)

    return (alpha / sigma) ** 2


def min_snr_weights(t, snr_gamma, prediction_type):
    """Per-sample Min-SNR-gamma weights as the training examples form them: min(snr, gamma), divided by snr for epsilon and by
    snr + 1 for v prediction (sample prediction: no division)."""
    snr = compute_snr(DDPMScheduler(), t)
    w = torch.stack([snr, snr_gamma * torch.ones_like(t)], dim=1).min(dim=1)[0]
    if prediction_type == "epsilon":
        return w / snr
    if prediction_type == "v_prediction":
        return w / (snr + 1)
    return w


def velocity(x0, noise, t):
    """the v_prediction target: DDPMScheduler.get_velocity(x0, noise, t)"""
    return DDPMScheduler(prediction_type="v_prediction").get_velocity(x0, noise, t)


def train_step_loss(sd, cfg, codes, noise, t, ids, mask=None, prediction_type="epsilon", snr_gamma=None):
    """ref_model.train_step_loss with the target of `prediction_type` (noise, x0 or the velocity) and, for snr_gamma not None,
    the training examples' Min-SNR-gamma weighting: mean over samples of w_b * the sample's MSE."""
    pred = ref_model.tts_forward(sd, cfg, ref_model.add_noise(codes, noise, t), t, ids, mask)
    target = {"epsilon": noise, "sample": codes}.get(prediction_type)
    if target is None:
        assert prediction_type == "v_prediction", prediction_type
        target = velocity(codes, noise, t)
    if snr_gamma is None:
        return F.mse_loss(pred.float(), target.float()), pred
    loss = F.mse_loss(pred.float(), target.float(), reduction="none")
    return (loss.mean(dim=list(range(1, len(loss.shape)))) * min_snr_weights(t, snr_gamma, prediction_type)).mean(), pred


def ddpm_step(model_output, t: int, x_t, noise, acp=None, n_infer=100, n_train=1000, prediction_type="epsilon"):
    """ref_model.ddpm_step (DDPMScheduler.step, clip_sample, fixed_small variance) for a model output of `prediction_type`"""
    if prediction_type == "epsilon":
        return ref_model.ddpm_step(model_output, t, x_t, noise, acp=acp, n_infer=n_infer, n_train=n_train)
    acp = ref_model.ddpm_alphas_cumprod(n_train) if acp is None else acp
    prev_t = t - n_train // n_infer
    a_t = acp[t]
    a_prev = acp[prev_t] if prev_t >= 0 else torch.tensor(1.0)
    b_t, b_prev = 1 - a_t, 1 - a_prev
    cur_alpha = a_t / a_prev
    cur_beta = 1 - cur_alpha
    if prediction_type == "sample":
        x0 = model_output.clamp(-1, 1)
    else:
        assert prediction_type == "v_prediction", prediction_type
        x0 = ((a_t ** 0.5) * x_t - (b_t ** 0.5) * model_output).clamp(-1, 1)
    mean = (a_prev ** 0.5 * cur_beta / b_t) * x0 + (cur_alpha ** 0.5 * b_prev / b_t) * x_t
    if t > 0:
        var = torch.clamp(b_prev / b_t * cur_beta, min=1e-20)
        mean = mean + var ** 0.5 * noise
    return mean
