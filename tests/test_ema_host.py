"""CPU: the EMA of the weights -- `FusedEMA`'s hyper-parameter validation and registration (before any device is needed), the argument
checks of pt_ema_prepare / pt_adamw_ema_step_dev / pt_ema_swap at the C ABI (no launch), and the diffusers 0.15 `EMAModel`
restatement the GPU tests compare against: its decay schedule at the corners and the rounding of its update."""
import math
import os
import sys

import numpy as np
import pytest
import torch

from util import ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))
from diffusers.training_utils import EMAModel  # noqa: E402


def _opt():
    from prompt_tts_b200.optim import FusedClipAdamW
    return FusedClipAdamW(None)         # never attached: nothing here may reach the stepper or a device


@pytest.mark.parametrize("kw", [dict(decay=1.5), dict(decay=-0.1), dict(decay=math.nan), dict(decay=math.inf), dict(decay="0.9"),
                                dict(decay=None), dict(decay=True), dict(decay=0.5, min_decay=0.6), dict(min_decay=-1e-3),
                                dict(min_decay=math.nan), dict(update_after_step=-1), dict(update_after_step=1.5),
                                dict(update_after_step=2.0), dict(update_after_step=True), dict(update_after_step="3"),
                                dict(use_ema_warmup=1), dict(use_ema_warmup="yes"), dict(inv_gamma=0.0), dict(inv_gamma=-1.0),
                                dict(inv_gamma=math.inf), dict(power=0.0), dict(power=-0.5), dict(power=math.nan)])
def test_bad_hyper_parameters_raise_before_registration(kw):
    from prompt_tts_b200.optim import FusedEMA
    opt = _opt()
    with pytest.raises(ValueError):
        FusedEMA(opt, **kw)
    assert opt.ema is None


@pytest.mark.parametrize("kw", [dict(), dict(decay=1.0, min_decay=1.0), dict(decay=0.0), dict(update_after_step=np.int64(5)),
                                dict(use_ema_warmup=True, inv_gamma=2, power=0.75), dict(decay=np.float32(0.999))])
def test_valid_hyper_parameters_register_once(kw):
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.optim import FusedEMA
    opt = _opt()
    ema = FusedEMA(opt, **kw)
    assert opt.ema is ema and ema.eflat is None and ema.optimization_step == 0 and ema.cur_decay is None
    with pytest.raises(_lib.PtError, match="already has an EMA"):
        FusedEMA(opt)
    assert opt.ema is ema


def test_defaults_are_diffusers():
    import inspect
    from prompt_tts_b200.optim import FusedEMA
    ours = inspect.signature(FusedEMA.__init__).parameters
    theirs = inspect.signature(EMAModel.__init__).parameters
    for k in ("decay", "min_decay", "update_after_step", "use_ema_warmup", "inv_gamma", "power"):
        assert ours[k].default == theirs[k].default, k


def test_ema_entry_points_validate_their_arguments():
    """Each call fails validation before anything is launched or dereferenced (no device needed)."""
    from prompt_tts_b200 import _lib, ops
    buf = torch.zeros(256)
    st = torch.zeros(16, dtype=torch.float64)
    p, z, s = ops._p(buf), ops._p(None), ops._p(st)

    def fused(*, pp=p, g=p, m=p, v=p, e=p, n=64, state=p, est=s):
        ops.call("adamw_ema_step_dev", pp, g, 0, m, v, z, e, n, state, est, z)

    def swap(*, pp=p, e=p, w=p, n=64):
        ops.call("ema_swap", pp, e, w, n, z)

    cases = [(lambda: ops.call("ema_prepare", z, z), "null state"),
             (lambda: fused(n=0), "n=0"), (lambda: fused(n=-4), "n=-4"), (lambda: fused(n=6), "n=6"),
             (lambda: fused(pp=z), "null"), (lambda: fused(g=z), "null"), (lambda: fused(m=z), "null"), (lambda: fused(v=z), "null"),
             (lambda: fused(e=z), "null"), (lambda: fused(state=z), "null"), (lambda: fused(est=z), "null"),
             (lambda: swap(n=0), "n=0"), (lambda: swap(n=-8), "n=-8"), (lambda: swap(n=10), "n=10"),
             (lambda: swap(pp=z), "null"), (lambda: swap(e=z), "null"), (lambda: swap(w=z), "null")]
    for fn, msg in cases:
        with pytest.raises(_lib.PtError, match=msg):
            fn()


def test_shim_decay_schedule_corners():
    d = EMAModel([], decay=0.9999).get_decay
    assert d(0) == 0.0 and d(1) == 0.0                       # the first update copies the weights (decay 0)
    assert d(2) == 2 / 11 and d(3) == 3 / 12                  # (1 + step) / (10 + step), step = optimization_step - 1
    assert d(10 ** 7) == 0.9999                               # capped at `decay`
    e = EMAModel([], decay=0.9, update_after_step=5).get_decay
    assert [e(k) for k in range(1, 7)] == [0.0] * 6 and e(7) == 2 / 11
    assert e(100) == 0.9
    m = EMAModel([], min_decay=0.5).get_decay
    assert m(1) == 0.0                                        # published 0.15: step <= 0 returns 0 before the clamps
    assert m(2) == 0.5 and m(3) == 0.5 and m(10) == 10 / 19   # raised to min_decay while (1 + step) / (10 + step) is below it
    w = EMAModel([], use_ema_warmup=True, inv_gamma=1.0, power=2 / 3).get_decay
    assert w(1) == 0.0 and w(2) == 1 - 2 ** (-2 / 3)
    assert w(1001) == 1 - (1 + 1000) ** (-2 / 3)
    w2 = EMAModel([], use_ema_warmup=True, inv_gamma=4.0, power=0.75, decay=0.99).get_decay
    assert w2(9) == 1 - (1 + 8 / 4.0) ** -0.75 and w2(10 ** 9) == 0.99


def test_shim_step_rounds_step_by_step():
    """torch's `s.sub_(c * (s - p))` is three fp32 roundings with c = float32(1 - decay); an FMA evaluation of the same update
    rounds differently on a measurable share of elements, so a kernel compiled with contraction would fail the GPU bit-equality."""
    rng = np.random.default_rng(0)
    n = 1 << 20
    s0 = rng.standard_normal(n).astype(np.float32)
    p = (s0 + rng.standard_normal(n).astype(np.float32) * np.float32(1e-2)).astype(np.float32)
    for decay in (2 / 11, 0.9999, 0.99):
        ema = EMAModel([torch.nn.Parameter(torch.from_numpy(s0.copy()))], decay=decay)
        ema.optimization_step = 10 ** 6                      # at the cap: decay = `decay`
        ema.step([torch.nn.Parameter(torch.from_numpy(p))])
        got = ema.shadow_params[0].numpy()
        c = np.float32(1 - ema.cur_decay_value)
        d = (s0 - p).astype(np.float32)
        want = (s0 - (c * d).astype(np.float32)).astype(np.float32)
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), decay
        fma = (s0.astype(np.float64) - np.float64(c) * d.astype(np.float64)).astype(np.float32)    # c * d is exact in double
        assert int((fma != want).sum()) > 0, decay
