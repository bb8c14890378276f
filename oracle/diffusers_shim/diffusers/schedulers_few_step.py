"""DDIMScheduler and DPMSolverMultistepScheduler, diffusers 0.15 semantics.

Not imported by the reference (which only trains with DDPMScheduler, train.py:8,32-36): these are the few-step schedulers a
user of the trained model swaps in for sampling (no retraining: same epsilon prediction, same linear-beta table).  Only the
options the product's samplers use are restated: epsilon prediction, linear betas; DPM-Solver++ of order 1 / 2 with the
midpoint solver, no thresholding.  Like the rest of this shim, parity with the real library is unpinned (no golden vectors
from diffusers exist offline).
"""
import numpy as np
import torch

from .schedulers import _Cfg


class SchedulerOutput:
    def __init__(self, prev_sample, pred_original_sample=None):
        self.prev_sample = prev_sample
        self.pred_original_sample = pred_original_sample


def _linear_alphas_cumprod(num_train_timesteps, beta_start, beta_end, beta_schedule, prediction_type):
    assert beta_schedule == "linear" and prediction_type == "epsilon"
    betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    return betas, torch.cumprod(1.0 - betas, dim=0)


class DDIMScheduler:
    """diffusers 0.15 DDIMScheduler: deterministic (eta = 0) to ancestral (eta = 1) steps on the training schedule."""

    def __init__(self, num_train_timesteps=1000, beta_start=1e-4, beta_end=0.02, beta_schedule="linear", clip_sample=True,
                 set_alpha_to_one=True, steps_offset=0, prediction_type="epsilon"):
        self.config = _Cfg(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                           beta_schedule=beta_schedule, clip_sample=clip_sample, set_alpha_to_one=set_alpha_to_one,
                           steps_offset=steps_offset, prediction_type=prediction_type)
        self.betas, self.alphas_cumprod = _linear_alphas_cumprod(num_train_timesteps, beta_start, beta_end, beta_schedule,
                                                                 prediction_type)
        self.alphas = 1.0 - self.betas
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(0, num_train_timesteps)[::-1].copy().astype(np.int64))

    def _get_variance(self, timestep, prev_timestep):
        alpha_prod_t = self.alphas_cumprod[timestep]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        beta_prod_t = 1 - alpha_prod_t
        beta_prod_t_prev = 1 - alpha_prod_t_prev
        return (beta_prod_t_prev / beta_prod_t) * (1 - alpha_prod_t / alpha_prod_t_prev)

    def set_timesteps(self, num_inference_steps, device=None):
        if num_inference_steps > self.config.num_train_timesteps:
            raise ValueError(f"num_inference_steps {num_inference_steps} > num_train_timesteps {self.config.num_train_timesteps}")
        self.num_inference_steps = num_inference_steps
        step_ratio = self.config.num_train_timesteps // self.num_inference_steps
        timesteps = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(timesteps).to(device)
        self.timesteps += self.config.steps_offset

    def step(self, model_output, timestep, sample, eta=0.0, use_clipped_model_output=False, generator=None,
             variance_noise=None, return_dict=True):
        timestep = int(timestep)
        prev_timestep = timestep - self.config.num_train_timesteps // self.num_inference_steps
        alpha_prod_t = self.alphas_cumprod[timestep]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        beta_prod_t = 1 - alpha_prod_t
        pred_original_sample = (sample - beta_prod_t ** 0.5 * model_output) / alpha_prod_t ** 0.5
        pred_epsilon = model_output
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


class DPMSolverMultistepScheduler:
    """diffusers 0.15 DPMSolverMultistepScheduler with algorithm_type "dpmsolver++", solver_type "midpoint" (orders 1 and 2)."""

    def __init__(self, num_train_timesteps=1000, beta_start=1e-4, beta_end=0.02, beta_schedule="linear", solver_order=2,
                 prediction_type="epsilon", thresholding=False, algorithm_type="dpmsolver++", solver_type="midpoint",
                 lower_order_final=True):
        assert solver_order in (1, 2) and not thresholding and algorithm_type == "dpmsolver++" and solver_type == "midpoint"
        self.config = _Cfg(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                           beta_schedule=beta_schedule, solver_order=solver_order, prediction_type=prediction_type,
                           thresholding=thresholding, algorithm_type=algorithm_type, solver_type=solver_type,
                           lower_order_final=lower_order_final)
        self.betas, self.alphas_cumprod = _linear_alphas_cumprod(num_train_timesteps, beta_start, beta_end, beta_schedule,
                                                                 prediction_type)
        self.alphas = 1.0 - self.betas
        self.alpha_t = torch.sqrt(self.alphas_cumprod)
        self.sigma_t = torch.sqrt(1 - self.alphas_cumprod)
        self.lambda_t = torch.log(self.alpha_t) - torch.log(self.sigma_t)
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.linspace(0, num_train_timesteps - 1, num_train_timesteps, dtype=np.float32)[::-1].copy())
        self.model_outputs = [None] * solver_order
        self.lower_order_nums = 0

    def set_timesteps(self, num_inference_steps, device=None):
        self.num_inference_steps = num_inference_steps
        timesteps = (np.linspace(0, self.config.num_train_timesteps - 1, num_inference_steps + 1)
                     .round()[::-1][:-1].copy().astype(np.int64))
        self.timesteps = torch.from_numpy(timesteps).to(device)
        self.model_outputs = [None] * self.config.solver_order
        self.lower_order_nums = 0

    def convert_model_output(self, model_output, timestep, sample):
        alpha_t, sigma_t = self.alpha_t[timestep], self.sigma_t[timestep]
        return (sample - sigma_t * model_output) / alpha_t

    def dpm_solver_first_order_update(self, model_output, timestep, prev_timestep, sample):
        lambda_t, lambda_s = self.lambda_t[prev_timestep], self.lambda_t[timestep]
        alpha_t = self.alpha_t[prev_timestep]
        sigma_t, sigma_s = self.sigma_t[prev_timestep], self.sigma_t[timestep]
        h = lambda_t - lambda_s
        return (sigma_t / sigma_s) * sample - (alpha_t * (torch.exp(-h) - 1.0)) * model_output

    def multistep_dpm_solver_second_order_update(self, model_output_list, timestep_list, prev_timestep, sample):
        t, s0, s1 = prev_timestep, timestep_list[-1], timestep_list[-2]
        m0, m1 = model_output_list[-1], model_output_list[-2]
        lambda_t, lambda_s0, lambda_s1 = self.lambda_t[t], self.lambda_t[s0], self.lambda_t[s1]
        alpha_t = self.alpha_t[t]
        sigma_t, sigma_s0 = self.sigma_t[t], self.sigma_t[s0]
        h, h_0 = lambda_t - lambda_s0, lambda_s0 - lambda_s1
        r0 = h_0 / h
        D0, D1 = m0, (1.0 / r0) * (m0 - m1)
        return ((sigma_t / sigma_s0) * sample
                - (alpha_t * (torch.exp(-h) - 1.0)) * D0
                - 0.5 * (alpha_t * (torch.exp(-h) - 1.0)) * D1)

    def step(self, model_output, timestep, sample, generator=None, return_dict=True):
        step_index = (self.timesteps == timestep).nonzero()
        step_index = len(self.timesteps) - 1 if len(step_index) == 0 else step_index.item()
        prev_timestep = 0 if step_index == len(self.timesteps) - 1 else int(self.timesteps[step_index + 1])
        lower_order_final = (step_index == len(self.timesteps) - 1) and self.config.lower_order_final and len(self.timesteps) < 15
        model_output = self.convert_model_output(model_output, timestep, sample)
        for i in range(self.config.solver_order - 1):
            self.model_outputs[i] = self.model_outputs[i + 1]
        self.model_outputs[-1] = model_output
        if self.config.solver_order == 1 or self.lower_order_nums < 1 or lower_order_final:
            prev_sample = self.dpm_solver_first_order_update(model_output, timestep, prev_timestep, sample)
        else:
            timestep_list = [int(self.timesteps[step_index - 1]), int(timestep)]
            prev_sample = self.multistep_dpm_solver_second_order_update(self.model_outputs, timestep_list, prev_timestep, sample)
        if self.lower_order_nums < self.config.solver_order:
            self.lower_order_nums += 1
        if not return_dict:
            return (prev_sample,)
        return SchedulerOutput(prev_sample)
