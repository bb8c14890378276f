"""EMAModel, diffusers 0.15 semantics (`diffusers.training_utils`).

Not imported by the reference: it is what diffusers' training scripts use under `--use_ema`, and the restatement that
`prompt_tts_b200.optim.FusedEMA` is checked against.  Only what that check needs is restated: the constructor's
hyper-parameters (no `model_cls` / `model_config`, no deprecated keyword names), `get_decay`, `step`, `copy_to`, `store`,
`restore` and `state_dict`.  Like the rest of this shim, parity with the real library is unpinned (no golden vectors from
diffusers exist offline).
"""
from typing import Iterable

import torch


class EMAModel:
    """Exponential moving average of a list of parameters."""

    def __init__(self, parameters: Iterable[torch.nn.Parameter], decay: float = 0.9999, min_decay: float = 0.0,
                 update_after_step: int = 0, use_ema_warmup: bool = False, inv_gamma: float = 1.0, power: float = 2 / 3):
        parameters = list(parameters)
        self.shadow_params = [p.clone().detach() for p in parameters]
        self.decay = decay
        self.min_decay = min_decay
        self.update_after_step = update_after_step
        self.use_ema_warmup = use_ema_warmup
        self.inv_gamma = inv_gamma
        self.power = power
        self.optimization_step = 0
        self.cur_decay_value = None
        self.temp_stored_params = None

    def get_decay(self, optimization_step: int) -> float:
        """Compute the decay factor for the exponential moving average."""
        step = max(0, optimization_step - self.update_after_step - 1)

        if step <= 0:
            return 0.0

        if self.use_ema_warmup:
            cur_decay_value = 1 - (1 + step / self.inv_gamma) ** -self.power
        else:
            cur_decay_value = (1 + step) / (10 + step)

        cur_decay_value = min(cur_decay_value, self.decay)
        # make sure decay is not smaller than min_decay
        cur_decay_value = max(cur_decay_value, self.min_decay)
        return cur_decay_value

    @torch.no_grad()
    def step(self, parameters: Iterable[torch.nn.Parameter]):
        parameters = list(parameters)

        self.optimization_step += 1

        # Compute the decay factor for the exponential moving average.
        decay = self.get_decay(self.optimization_step)
        self.cur_decay_value = decay
        one_minus_decay = 1 - decay

        for s_param, param in zip(self.shadow_params, parameters):
            if param.requires_grad:
                s_param.sub_(one_minus_decay * (s_param - param))
            else:
                s_param.copy_(param)

    def copy_to(self, parameters: Iterable[torch.nn.Parameter]) -> None:
        """Copy the current averaged parameters into the given collection of parameters."""
        parameters = list(parameters)
        for s_param, param in zip(self.shadow_params, parameters):
            param.data.copy_(s_param.to(param.device).data)

    def store(self, parameters: Iterable[torch.nn.Parameter]) -> None:
        """Save the current parameters (on the host) for restoring later."""
        self.temp_stored_params = [param.detach().cpu().clone() for param in parameters]

    def restore(self, parameters: Iterable[torch.nn.Parameter]) -> None:
        """Restore the parameters stored with the `store` method."""
        if self.temp_stored_params is None:
            raise RuntimeError("This ExponentialMovingAverage has no `store()`ed weights to `restore()`")
        for c_param, param in zip(self.temp_stored_params, parameters):
            param.data.copy_(c_param.data)
        self.temp_stored_params = None

    def state_dict(self) -> dict:
        return {
            "decay": self.decay,
            "min_decay": self.min_decay,
            "optimization_step": self.optimization_step,
            "update_after_step": self.update_after_step,
            "use_ema_warmup": self.use_ema_warmup,
            "inv_gamma": self.inv_gamma,
            "power": self.power,
            "shadow_params": self.shadow_params,
        }
