"""The reference's optimiser lines (train.py:41-47 AdamW(lr 1e-5, betas (0.95, 0.999), weight_decay 1e-6, eps 1e-8);
train.py:116-120 clip_grad_norm_(1.0) -> step -> zero_grad) as three kernels over flat buffers (SURVEY 8f rank 1).

`DenoiserTrainStep` leaves all gradients of a step in one flat fp32 buffer (dp.GradSync, laid out in the order the backward
sweep completes them, all-reduced in place).  `FusedClipAdamW` keeps, in that same layout,
    pflat  fp32 master parameters -- every `nn.Parameter` becomes a view of it (k=3 conv weights a permuted view of their tap-major
           storage), so `state_dict()`, checkpoints and the module tree are unchanged;
    m, v   AdamW moments;
    wflat  the bf16 shadow of pflat -- the GEMM weight operands (`engine.PackCache` static entries) are views of it, written by
           the AdamW kernel itself, so there is no fp32 -> bf16 re-pack pass after an update (round 1: 292 launches, 3.2 GB).
A step is: sum of squares of the gradient buffer -> `pt_adamw_prepare` (one thread: step += 1, bias corrections, clip factor,
all in DEVICE memory) -> one elementwise AdamW kernel.  No host value is baked into a launch: the step counter, the learning
rate and the clip factor are read from device memory, so a CUDA graph that captured `step()` replays the reference's optimiser
exactly (`tests/test_optim_gpu.py::test_fused_adamw_graph_replays`).  Parameters that never receive a gradient (the 32 dead
`proj_out` tensors) are left untouched, as torch.optim.AdamW does for `grad is None`.

`FusedEMA` adds diffusers' EMAModel (the average LDM-style models are sampled from): with one registered, a step is four
launches, the fourth the same AdamW kernel also updating the average.
"""
from __future__ import annotations

import collections
import contextlib
import math
import numbers
from typing import Dict, Optional

import torch

from . import ops

# slots of the device-side state (include/prompt_tts_b200.h)
LR, BETA1, BETA2, EPS, WD, MAX_NORM, GSCALE, STEP, CLIP, STEP_SIZE, INV_SQRT_BC2, DECAY, GNORM, GNORM_SQ, NSTATE = 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 16
NPARTS = 1184      # blocks of the deterministic norm reduction (8 per SM)


class FusedClipAdamW:
    def __init__(self, stepper, lr: float = 1e-5, betas=(0.95, 0.999), weight_decay: float = 1e-6, eps: float = 1e-8,
                 max_norm: float = 1.0):
        self.stepper = stepper
        self.lr, self.betas, self.wd, self.eps, self.max_norm = lr, betas, weight_decay, eps, max_norm
        self.pflat = self.m = self.v = self.wflat = self.partials = self.state = None
        self.ema = None       # a FusedEMA registers itself here; step() then also updates it

    # ------------------------------------------------------------------------------------------ flat state
    def attach(self) -> None:
        """Build the flat master / moment / shadow buffers (needs the gradient layout: run one DenoiserTrainStep first) and
        re-home every parameter into the master buffer.  Called by the first `step()`; call it earlier to capture a step whose
        GEMMs already read the shadow."""
        if self.pflat is not None:
            return
        gs = self.stepper.grad_sync
        if gs is None or gs.layout is None:
            raise ops._lib.PtError("FusedClipAdamW: run one DenoiserTrainStep first (it defines the flat gradient layout)")
        dev = gs.flat.device
        self.pflat = torch.zeros(gs.total, dtype=torch.float32, device=dev)
        self.wflat = torch.zeros(gs.total, dtype=torch.bfloat16, device=dev)
        cache = self.stepper.cache
        for params, off, n, kind in gs.groups:
            sl = self.pflat[off:off + n]
            if kind == "conv":
                (p,) = params
                Co, Ci, k = p.shape
                packed = sl.view(Co, k, Ci)
                packed.copy_(p.data.permute(0, 2, 1))
                p.data = packed.permute(0, 2, 1)           # logical [Co, Ci, k]; storage tap-major = the GEMM layout
                cache.add_static("conv", params, self.wflat[off:off + n].view(Co, k * Ci), self._refresher(off, n))
                continue
            o = off
            for p in params:
                kk = p.numel()
                self.pflat[o:o + kk].copy_(p.data.reshape(-1))
                p.data = self.pflat[o:o + kk].view(p.shape)       # the module tree now reads / checkpoints the master buffer
                o += kk
            assert o == off + n
            p0 = params[0]
            if p0.dim() >= 2:
                rows = sum(p.shape[0] for p in params)
                cache.add_static("lin", params, self.wflat[off:off + n].view(rows, n // rows), self._refresher(off, n))
            elif p0.dim() == 1 and len(params) > 1:
                cache.add_static("bias", params, self.pflat[off:off + n], None)
        ops.cast_bf16(self.pflat, self.wflat)
        self.m = torch.zeros_like(self.pflat)
        self.v = torch.zeros_like(self.pflat)
        self.partials = torch.zeros(NPARTS, dtype=torch.float32, device=dev)
        host = [0.0] * NSTATE
        host[LR], host[BETA1], host[BETA2], host[EPS], host[WD], host[MAX_NORM], host[GSCALE] = (
            self.lr, self.betas[0], self.betas[1], self.eps, self.wd, self.max_norm if self.max_norm else 0.0, 1.0)
        self.state = torch.tensor(host, dtype=torch.float32, device=dev)       # slot STEP = int32 0
        if gs.comm is not None:
            gs.cast_back = False          # the AdamW kernel reads the averaged bf16 gradients directly
        if self.ema is not None:
            self.ema._init_shadow()

    def _refresher(self, off: int, n: int):
        def refresh():      # a parameter of this group was written from outside (load_state_dict, p.data.copy_)
            ops.cast_bf16(self.pflat[off:off + n], self.wflat[off:off + n])
        return refresh

    def sync_shadow(self) -> None:
        """Re-derive the whole bf16 shadow from the fp32 masters."""
        ops.cast_bf16(self.pflat, self.wflat)

    # ------------------------------------------------------------------------------------------ hyper-parameters (device side)
    def set_lr(self, lr: float) -> None:
        """What an LR scheduler calls (train.py:60-65,119): a device write, valid between replays of a captured step."""
        self.lr = lr
        if self.state is not None:
            self.state[LR:LR + 1].fill_(lr)

    @property
    def step_count(self) -> int:
        return 0 if self.state is None else int(self.state[STEP:STEP + 1].view(torch.int32).item())

    # ------------------------------------------------------------------------------------------ step
    @torch.no_grad()
    def step(self) -> torch.Tensor:
        """Clip to max_norm (global L2 norm over all gradients, like clip_grad_norm_) and apply AdamW in place.
        Returns the squared gradient norm as a 0-d device tensor (no synchronisation).  A no-op on micro-steps that do not
        synchronise gradients (accelerate's optimizer wrapper under `accumulate`, train.py:80,118)."""
        self.attach()
        if self.ema is not None and self.ema.is_swapped:
            raise ops._lib.PtError("FusedClipAdamW.step: the EMA weights are swapped in; leave `FusedEMA.swapped()` first")
        if not getattr(self.stepper, "sync_gradients", True):
            return self.gnorm_sq
        gs = self.stepper.grad_sync
        g_bf16 = gs.comm is not None and not gs.cast_back
        # global norm, deterministically (identical gradients -> bit-identical clip factor on every rank: replicas never drift apart)
        ops.call("sumsq_partials", ops._p(gs.comm if g_bf16 else gs.flat), 1 if g_bf16 else 0, gs.total, ops._p(self.partials), NPARTS, ops._stream())
        ops.call("adamw_prepare_det", ops._p(self.state), ops._p(self.partials), NPARTS, ops._stream())
        if self.ema is None:
            ops.call("adamw_step_dev", ops._p(self.pflat), ops._p(gs.comm if g_bf16 else gs.flat), 1 if g_bf16 else 0, ops._p(self.m),
                     ops._p(self.v), ops._p(self.wflat), gs.total, ops._p(self.state), ops._stream())
        else:
            ops.call("ema_prepare", ops._p(self.ema.state), ops._stream())
            ops.call("adamw_ema_step_dev", ops._p(self.pflat), ops._p(gs.comm if g_bf16 else gs.flat), 1 if g_bf16 else 0,
                     ops._p(self.m), ops._p(self.v), ops._p(self.wflat), ops._p(self.ema.eflat), gs.total, ops._p(self.state),
                     ops._p(self.ema.state), ops._stream())
        return self.gnorm_sq

    @property
    def gnorm_sq(self) -> torch.Tensor:
        """Squared global gradient norm of the last step (0-d device tensor, no synchronisation)."""
        return self.state[GNORM_SQ]

    # ------------------------------------------------------------------------------------------ checkpoints (train.py:141-143)
    def state_dict(self) -> Dict[str, torch.Tensor]:
        self.attach()
        return {"state": self.state.clone(), "m": self.m.clone(), "v": self.v.clone(),
                "layout": [(off, n, kind) for _, off, n, kind in self.stepper.grad_sync.groups]}

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        self.attach()
        want = [(off, n, kind) for _, off, n, kind in self.stepper.grad_sync.groups]
        if list(map(tuple, sd["layout"])) != want:
            raise ops._lib.PtError("FusedClipAdamW.load_state_dict: the checkpoint was written for a different flat layout")
        self.state.copy_(sd["state"])
        self.m.copy_(sd["m"])
        self.v.copy_(sd["v"])
        self.lr = float(self.state[LR].item())
        self.sync_shadow()


# slots of the EMA's float64 device state (include/prompt_tts_b200.h PT_EMA_*)
EMA_DECAY, EMA_MIN_DECAY, EMA_UPDATE_AFTER, EMA_USE_WARMUP, EMA_INV_GAMMA, EMA_POWER, EMA_STEP, EMA_CUR_DECAY, EMA_COEF, EMA_NSTATE = (
    0, 1, 2, 3, 4, 5, 6, 7, 8, 16)


def _real(name: str, x) -> float:
    if isinstance(x, bool) or not isinstance(x, numbers.Real) or not math.isfinite(float(x)):
        raise ValueError(f"FusedEMA: {name}={x!r} must be a finite real number")
    return float(x)


class FusedEMA:
    """Exponential moving average of the weights that `opt` trains: diffusers 0.15 `training_utils.EMAModel` (its defaults, its
    decay schedule, its fp32 update rounded step by step), updated inside the AdamW kernel of every optimiser step.

    The average is one flat fp32 buffer `eflat` in the optimiser's layout plus a float64 device state (hyper-parameters, the
    optimisation step, the current decay), so a CUDA graph that captured `stepper(); opt.step()` replays as the next EMA step too.
    It steps once per optimiser update and sees the weights after that update (`optimizer.step(); ema.step(...)`); micro-steps of an
    accumulation window, where `opt.step()` is a no-op, do not step it.

    The average starts from the master weights: at construction if `opt` is already attached, otherwise when `opt.attach()` runs
    (its first `step()`).  That equals diffusers' copy at construction unless the weights are written in between.  Parameters
    outside the flat layout (the never-trained `proj_out` tensors) keep, as diffusers' update keeps them, the value they had then.
    """

    def __init__(self, opt: FusedClipAdamW, decay: float = 0.9999, min_decay: float = 0.0, update_after_step: int = 0,
                 use_ema_warmup: bool = False, inv_gamma: float = 1.0, power: float = 2 / 3):
        decay, min_decay = _real("decay", decay), _real("min_decay", min_decay)
        if not 0.0 <= min_decay <= decay <= 1.0:
            raise ValueError(f"FusedEMA: need 0 <= min_decay ({min_decay}) <= decay ({decay}) <= 1")
        if isinstance(update_after_step, bool) or not isinstance(update_after_step, numbers.Integral) or update_after_step < 0:
            raise ValueError(f"FusedEMA: update_after_step={update_after_step!r} must be an integer >= 0")
        if not isinstance(use_ema_warmup, bool):
            raise ValueError(f"FusedEMA: use_ema_warmup={use_ema_warmup!r} must be a bool")
        inv_gamma, power = _real("inv_gamma", inv_gamma), _real("power", power)
        if inv_gamma <= 0.0 or power <= 0.0:
            raise ValueError(f"FusedEMA: inv_gamma ({inv_gamma}) and power ({power}) must be > 0")
        if getattr(opt, "ema", None) is not None:
            raise ops._lib.PtError("FusedEMA: this optimiser already has an EMA")
        self.opt = opt
        self.decay, self.min_decay, self.update_after_step = decay, min_decay, int(update_after_step)
        self.use_ema_warmup, self.inv_gamma, self.power = bool(use_ema_warmup), inv_gamma, power
        self.eflat = self.state = None
        self.is_swapped = False
        self.frozen: Dict[str, torch.Tensor] = {}      # parameters outside the flat layout, as they were when the average started
        opt.ema = self
        if opt.pflat is not None:
            self._init_shadow()

    def _init_shadow(self) -> None:
        opt = self.opt
        self.eflat = opt.pflat.clone()
        host = [0.0] * EMA_NSTATE
        host[EMA_DECAY], host[EMA_MIN_DECAY], host[EMA_UPDATE_AFTER] = self.decay, self.min_decay, float(self.update_after_step)
        host[EMA_USE_WARMUP], host[EMA_INV_GAMMA], host[EMA_POWER] = float(self.use_ema_warmup), self.inv_gamma, self.power
        self.state = torch.tensor(host, dtype=torch.float64, device=opt.pflat.device)
        self.frozen = {k: v.detach().clone() for k, v in self._params().items() if not self._in_flat(v)}

    def _params(self) -> Dict[str, torch.Tensor]:
        return {k: v for k, v in self.opt.stepper.model.state_dict(keep_vars=True).items() if isinstance(v, torch.nn.Parameter)}

    def _in_flat(self, p: torch.Tensor) -> bool:
        return p.untyped_storage().data_ptr() == self.opt.pflat.untyped_storage().data_ptr()

    def _attached(self) -> None:
        if self.is_swapped:
            raise ops._lib.PtError("FusedEMA: the EMA weights are swapped in; leave `swapped()` first")
        self.opt.attach()         # defines the layout (raises before the first DenoiserTrainStep) and starts the average

    # ------------------------------------------------------------------------------------------ diffusers' attributes
    @property
    def optimization_step(self) -> int:
        """Optimiser updates the average has seen (synchronises)."""
        return 0 if self.state is None else int(self.state[EMA_STEP].item())

    @property
    def cur_decay(self) -> Optional[torch.Tensor]:
        """Decay of the last update as a 0-d float64 device tensor (no synchronisation); None before the average starts."""
        return None if self.state is None else self.state[EMA_CUR_DECAY]

    # ------------------------------------------------------------------------------------------ evaluation with the EMA weights
    def _swap(self) -> None:
        opt = self.opt
        ops.call("ema_swap", ops._p(opt.pflat), ops._p(self.eflat), ops._p(opt.wflat), opt.pflat.numel(), ops._stream())
        opt.stepper.cache.epoch += 1      # no pack of a swapped parameter made outside the static shadow survives

    @contextlib.contextmanager
    def swapped(self):
        """Within the block the model's weights (fp32 masters and their bf16 shadow) are the EMA, and the EMA buffer holds the
        trained weights; both are exchanged back on exit.  No buffer is reallocated, so a training step captured in a CUDA graph
        before the block replays correctly after it.  (diffusers: store(); copy_to(); ...; restore(), without the host copy.)"""
        if torch.cuda.is_current_stream_capturing():
            raise ops._lib.PtError("FusedEMA.swapped: not available while the current stream is being captured")
        self._attached()
        self._swap()
        self.is_swapped = True
        try:
            yield self
        finally:
            self.is_swapped = False
            self._swap()

    def copy_to(self) -> None:
        """Make the EMA the model's weights for good (diffusers' copy_to before saving); the average itself is unchanged."""
        self._attached()
        self.opt.pflat.copy_(self.eflat)
        self.opt.sync_shadow()
        self.opt.stepper.cache.epoch += 1
        params = self._params()
        for k, v in self.frozen.items():
            params[k].data.copy_(v)

    def model_state_dict(self) -> Dict[str, torch.Tensor]:
        """The EMA weights in the model's own format: the keys, shapes and order of `model.state_dict()`, loadable with strict=True.
        Buffers come from the model."""
        self._attached()
        out = collections.OrderedDict()
        for k, v in self.opt.stepper.model.state_dict(keep_vars=True).items():
            if not isinstance(v, torch.nn.Parameter):
                t = v.detach()
            elif k in self.frozen:
                t = self.frozen[k]
            else:       # every trained parameter's storage is a view of pflat: the same view of eflat is its average
                t = torch.as_strided(self.eflat, v.shape, v.stride(), v.storage_offset())
            out[k] = t.clone(memory_format=torch.contiguous_format)
        return out

    # ------------------------------------------------------------------------------------------ checkpoints (resume)
    def state_dict(self) -> Dict[str, object]:
        self._attached()
        return {"state": self.state.clone(), "eflat": self.eflat.clone(), "frozen": {k: v.clone() for k, v in self.frozen.items()},
                "layout": [(off, n, kind) for _, off, n, kind in self.opt.stepper.grad_sync.groups]}

    def load_state_dict(self, sd: Dict[str, object]) -> None:
        self._attached()
        want = [(off, n, kind) for _, off, n, kind in self.opt.stepper.grad_sync.groups]
        if list(map(tuple, sd["layout"])) != want or set(sd["frozen"]) != set(self.frozen):
            raise ops._lib.PtError("FusedEMA.load_state_dict: the checkpoint was written for a different flat layout")
        self.state.copy_(sd["state"])
        self.eflat.copy_(sd["eflat"])
        for k, v in sd["frozen"].items():
            self.frozen[k].copy_(v)
        h = self.state.tolist()
        self.decay, self.min_decay, self.update_after_step = h[EMA_DECAY], h[EMA_MIN_DECAY], int(h[EMA_UPDATE_AFTER])
        self.use_ema_warmup, self.inv_gamma, self.power = bool(h[EMA_USE_WARMUP]), h[EMA_INV_GAMMA], h[EMA_POWER]
