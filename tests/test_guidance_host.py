"""CPU: classifier-free guidance -- `guidance_scale` validation in all three samplers (before any device is needed), the
`cond_keep` checks, and the argument checks of pt_cond_select_bf16 / pt_cfg_combine / pt_rows_add_bias_bf16 at the C ABI (no
launch)."""
import math

import numpy as np
import pytest
import torch

from util import load_cfg


@pytest.fixture(scope="module")
def cpu_model():
    from prompt_tts_b200.models import TTSSingleSpeaker
    return TTSSingleSpeaker(load_cfg("tiny"))


def _samplers(model):
    from prompt_tts_b200.sample import DDIMSampler, DDPMSampler, DPMSolverSampler
    return [DDPMSampler(model, n_infer=2), DDIMSampler(model, n_infer=2, eta=1.0), DPMSolverSampler(model, n_infer=2)]


@pytest.mark.parametrize("bad", [True, False, float("nan"), float("inf"), -float("inf"), 0.99, 0.0, -3.0, "3", None, 1 + 0j,
                                 torch.tensor(3.0)])
def test_guidance_scale_is_validated_first(cpu_model, bad):
    """ValueError from every sampler, even though the inputs are CPU tensors (which fail later, with PtError)"""
    for smp in _samplers(cpu_model):
        with pytest.raises(ValueError, match="guidance_scale"):
            smp.sample(torch.zeros(1, 24, dtype=torch.int32), 16, guidance_scale=bad)


@pytest.mark.parametrize("ok", [1, 1.0, 3, 7.5, np.float32(2.0), np.float64(1.0), 1e6])
def test_valid_guidance_scale_reaches_the_device_check(cpu_model, ok):
    from prompt_tts_b200 import _lib
    for smp in _samplers(cpu_model):
        with pytest.raises(_lib.PtError, match="CUDA"):
            smp.sample(torch.zeros(1, 24, dtype=torch.int32), 16, guidance_scale=ok)


def test_guidance_default_is_unguided():
    import inspect
    from prompt_tts_b200.sample import _Sampler
    assert inspect.signature(_Sampler.sample).parameters["guidance_scale"].default == 1.0


def test_cond_keep_is_keyword_only_and_off_by_default():
    import inspect
    from prompt_tts_b200.models import TTSSingleSpeaker
    from prompt_tts_b200.train import DenoiserTrainStep
    p = inspect.signature(TTSSingleSpeaker.forward).parameters["cond_keep"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is None
    assert list(inspect.signature(TTSSingleSpeaker.forward).parameters)[-1] == "cond_keep"
    assert inspect.signature(DenoiserTrainStep.__call__).parameters["cond_keep"].default is None


def test_cond_keep_mask_rejects_bad_masks():
    from prompt_tts_b200 import _lib
    from prompt_tts_b200 import engine as E
    for bad in (torch.ones(4, dtype=torch.bool), torch.ones(3, dtype=torch.bool), torch.ones(4, 1, dtype=torch.uint8),
                torch.ones(4, dtype=torch.float32), torch.ones(4, dtype=torch.int64), [1, 1, 1, 1], None):
        with pytest.raises(_lib.PtError, match="cond_keep"):      # CPU, wrong shape, wrong dtype, not a tensor
            E.cond_keep_mask(bad, 4, torch.device("cuda", 0), "test")


def test_guidance_entry_points_validate_their_arguments():
    """Each call fails validation before anything is launched or dereferenced (no device needed)."""
    from prompt_tts_b200 import _lib, ops
    buf = torch.zeros(256)
    keep = torch.ones(8, dtype=torch.uint8)
    p, z, k = ops._p(buf), ops._p(None), ops._p(keep)
    odd = buf.data_ptr() + 2                        # not 16-byte aligned

    def sel(*, x=p, keep=k, y=p, B=2, per=64):
        ops.call("cond_select_bf16", x, keep, y, B, per, z)

    def cfg(*, e=p, o=p, n=64, w=3.0):
        ops.call("cfg_combine", e, o, n, w, z)

    def rab(*, r=p, b=p, y=p, rows=4, C=16):
        ops.call("rows_add_bias_bf16", r, b, y, rows, C, z)

    cases = [(lambda: sel(B=0), "B=0"), (lambda: sel(B=-1), "B=-1"), (lambda: sel(per=0), "per_sample=0"),
             (lambda: sel(per=12), "per_sample=12"), (lambda: sel(keep=z), "keep"), (lambda: sel(x=z), "required"),
             (lambda: sel(x=odd), "aligned"), (lambda: sel(y=odd), "aligned"),
             (lambda: cfg(n=0), "n=0"), (lambda: cfg(n=-5), "n=-5"), (lambda: cfg(e=z), "required"),
             (lambda: cfg(w=math.nan), "finite"), (lambda: cfg(w=math.inf), "finite"), (lambda: cfg(w=-math.inf), "finite"),
             (lambda: rab(rows=0), "rows=0"), (lambda: rab(C=12), "C=12"), (lambda: rab(C=0), "C=0"), (lambda: rab(b=z), "required"),
             (lambda: rab(r=odd), "aligned"), (lambda: rab(y=odd), "aligned")]
    for fn, msg in cases:
        with pytest.raises(_lib.PtError, match=msg):
            fn()
