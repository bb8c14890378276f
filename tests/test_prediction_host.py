"""CPU: sample / v prediction and Min-SNR-gamma weighting -- `prediction_type` / `snr_gamma` validation in the train step and all
three samplers (before any device is needed), the defaults, the argument checks of pt_diffusion_loss and the `_pred` step entry
points at the C ABI (no launch), and the oracle's restated branches (tests/prediction_oracle.py): per-step identities between the three parameterisations of
one model output, `get_velocity`, `compute_snr`, and the loops on a Gaussian target whose predictors are known in closed form."""
import inspect
import math

import numpy as np
import pytest
import torch

from prediction_oracle import DDIMScheduler, DDPMScheduler, DPMSolverMultistepScheduler, compute_snr
from util import load_cfg, rel

PRED_TYPES = ("epsilon", "sample", "v_prediction")


@pytest.fixture(scope="module")
def cpu_model():
    from prompt_tts_b200.models import TTSSingleSpeaker
    return TTSSingleSpeaker(load_cfg("tiny"))


def _sampler_classes():
    from prompt_tts_b200.sample import DDIMSampler, DDPMSampler, DPMSolverSampler
    return [DDPMSampler, DDIMSampler, DPMSolverSampler]


# ---------------------------------------------------------------------------------------------------------------- Python API
@pytest.mark.parametrize("bad", [None, True, 0, 1, 2, "eps", "EPSILON", "v", "v-prediction", "x0", "", b"epsilon", ["sample"],
                                 float("nan")])
def test_prediction_type_is_validated_first(cpu_model, bad):
    """ValueError from every constructor, before the train step builds its flat gradient buffer on the device"""
    from prompt_tts_b200.train import DenoiserTrainStep
    for cls in _sampler_classes():
        with pytest.raises(ValueError, match="prediction_type"):
            cls(cpu_model, prediction_type=bad)
    with pytest.raises(ValueError, match="prediction_type"):
        DenoiserTrainStep(cpu_model, prediction_type=bad)


@pytest.mark.parametrize("bad", [True, False, float("nan"), float("inf"), -float("inf"), 0, 0.0, -0.0, -1.0, -5, "5", 1 + 0j,
                                 torch.tensor(5.0), [5.0]])
def test_snr_gamma_is_validated_first(cpu_model, bad):
    from prompt_tts_b200.train import DenoiserTrainStep
    for pt in PRED_TYPES:
        with pytest.raises(ValueError, match="snr_gamma"):
            DenoiserTrainStep(cpu_model, prediction_type=pt, snr_gamma=bad)


@pytest.mark.parametrize("ok", [1, 5, 5.0, 0.5, 1e-3, np.float32(5.0), np.float64(20.0), np.int64(3)])
def test_valid_snr_gamma_is_accepted(ok):
    from prompt_tts_b200 import ops
    for pt in PRED_TYPES:
        assert ops.check_prediction("test", pt, ok) == (ops.PRED_TYPES[pt], float(ok))
    assert ops.check_prediction("test", "epsilon") == (0, 0.0)
    assert ops.PRED_TYPES == {"epsilon": 0, "sample": 1, "v_prediction": 2}      # PT_PRED_* of the header


@pytest.mark.parametrize("pt", PRED_TYPES)
def test_valid_prediction_type_reaches_the_device_check(cpu_model, pt):
    from prompt_tts_b200 import _lib
    for cls in _sampler_classes():
        smp = cls(cpu_model, n_infer=2, prediction_type=pt)
        assert smp.prediction_type == pt
        with pytest.raises(_lib.PtError, match="CUDA"):
            smp.sample(torch.zeros(1, 24, dtype=torch.int32), 16)


def test_defaults_are_epsilon_and_keyword_only():
    from prompt_tts_b200.train import DenoiserTrainStep
    sigs = [inspect.signature(c.__init__) for c in _sampler_classes() + [DenoiserTrainStep]]
    for sig in sigs:
        p = sig.parameters["prediction_type"]
        assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default == "epsilon"
    p = inspect.signature(DenoiserTrainStep.__init__).parameters["snr_gamma"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is None
    assert list(inspect.signature(DenoiserTrainStep.__init__).parameters)[:4] == ["self", "model", "grad_sync", "accumulation_steps"]
    for cls in _sampler_classes():
        assert "snr_gamma" not in inspect.signature(cls.__init__).parameters


# ---------------------------------------------------------------------------------------------------------------- C ABI
def test_prediction_entry_points_validate_their_arguments():
    """Each call fails validation before anything is launched or dereferenced (no device needed)."""
    from prompt_tts_b200 import _lib, ops
    buf = torch.zeros(256)
    p, z = ops._p(buf), ops._p(None)

    def loss(*, ptrs=(p,) * 8, B=2, per=64, pt=2, g=5.0, gs=1.0):
        ops.call("diffusion_loss", *ptrs, B, per, pt, g, gs, z)

    def ddpm(*, pt=1, n=64, T=16, keep=0, a=0.5, ap=0.6):
        ops.call("ddpm_step_pred", p, p, p, z, p, n, T, keep, a, ap, pt, z)

    def ddim(*, pt=1, n=64, eta=0.0, a=0.5):
        ops.call("ddim_step_pred", p, p, p, z, z, p, n, 16, 0, a, 0.6, eta, 1.0, 0.0, pt, z)

    def dpmpp(*, pt=2, order=2, m_prev=p, s0=0.5):
        ops.call("dpmpp_step_pred", p, p, m_prev, p, z, z, p, 64, 16, 0, s0, 0.4, 0.6, order, 1.0, 0.0, pt, z)

    cases = [(lambda: loss(pt=3), "pred_type=3"), (lambda: loss(pt=-1), "pred_type=-1"), (lambda: loss(g=-1.0), "snr_gamma"),
             (lambda: loss(g=math.nan), "snr_gamma"), (lambda: loss(g=math.inf), "snr_gamma"), (lambda: loss(B=0), "B=0"),
             (lambda: loss(B=-3), "B=-3"), (lambda: loss(per=0), "per_sample=0")]
    for k in range(8):                               # pred, x0, noise, t, sqrt_acp, sqrt_1macp, loss, dpred
        cases.append((lambda k=k: loss(ptrs=tuple(z if j == k else p for j in range(8))), "null pointer"))
    cases += [(lambda: ddpm(pt=3), "pred_type=3"), (lambda: ddpm(pt=-1), "pred_type=-1"), (lambda: ddpm(n=0), "n=0"),
              (lambda: ddpm(keep=17), "keep=17"), (lambda: ddpm(a=0.0), "acp_t"), (lambda: ddpm(ap=0.4), "acp_prev"),
              (lambda: ddim(pt=7), "pred_type=7"), (lambda: ddim(n=60), "n=60"), (lambda: ddim(eta=-1.0), "eta"),
              (lambda: ddim(a=1.0), "acp_t"),
              (lambda: dpmpp(pt=3), "pred_type=3"), (lambda: dpmpp(order=3), "order=3"), (lambda: dpmpp(m_prev=z), "order=2"),
              (lambda: dpmpp(s0=0.7), "acp_t")]
    for fn, msg in cases:
        with pytest.raises(_lib.PtError, match=msg):
            fn()


# ---------------------------------------------------------------------------------------------------------------- oracle
def _scheds(pt):
    return {"ddpm": DDPMScheduler(prediction_type=pt), "ddim": DDIMScheduler(prediction_type=pt),
            "dpm": DPMSolverMultistepScheduler(prediction_type=pt)}


def _convert(eps, x, a, pt):
    """the exact x0 / v forms, in float64, of an epsilon output at (x, alphas_cumprod a)"""
    a = a.double()
    x0 = (x.double() - (1 - a).sqrt() * eps.double()) / a.sqrt()
    out = {"epsilon": eps.double(), "sample": x0, "v_prediction": a.sqrt() * eps.double() - (1 - a).sqrt() * x0}[pt]
    return out.float()


@pytest.mark.parametrize("t", [990, 500, 100, 20, 0])
def test_oracle_ddpm_and_ddim_steps_agree_across_parameterisations(t):
    g = torch.Generator().manual_seed(t)
    x, eps, nz = (torch.randn(4, 8, 64, generator=g) for _ in range(3))
    for kind, step in [("ddpm", lambda s, o: s.step(o, t, x, noise=nz)),
                       ("ddim_eta0", lambda s, o: s.step(o, t, x, eta=0.0).prev_sample),
                       ("ddim_eta1", lambda s, o: s.step(o, t, x, eta=1.0, variance_noise=nz).prev_sample)]:
        res = {}
        for pt in PRED_TYPES:
            s = _scheds(pt)["ddpm" if kind == "ddpm" else "ddim"]
            s.set_timesteps(50)
            res[pt] = step(s, _convert(eps, x, s.alphas_cumprod[t], pt))
        for pt in ("sample", "v_prediction"):
            assert rel(res[pt], res["epsilon"]) <= 1e-5, (kind, t, pt, rel(res[pt], res["epsilon"]))


@pytest.mark.parametrize("n", [20, 5])
def test_oracle_dpm_solver_agrees_across_parameterisations(n):
    """a whole DPM-Solver++ loop: first-order first step, second-order steps from the history, (n = 5) first-order last step"""
    g = torch.Generator().manual_seed(n)
    x_T = torch.randn(4, 8, 64, generator=g)
    res = {}
    for pt in PRED_TYPES:
        s = _scheds(pt)["dpm"]
        s.set_timesteps(n)
        x = x_T.clone()
        for t in s.timesteps.tolist():
            eps = torch.tanh(x) * 0.9 + 0.1 * torch.sin(3.0 * x)     # a fixed smooth "model"
            x = s.step(_convert(eps, x, s.alphas_cumprod[t], pt), t, x).prev_sample
        res[pt] = x
    for pt in ("sample", "v_prediction"):
        assert rel(res[pt], res["epsilon"]) <= 1e-5, (n, pt, rel(res[pt], res["epsilon"]))


def test_get_velocity_is_its_formula():
    import prediction_oracle as po
    s = DDPMScheduler(prediction_type="v_prediction")
    g = torch.Generator().manual_seed(3)
    x0, nz = torch.randn(6, 8, 32, generator=g), torch.randn(6, 8, 32, generator=g)
    t = torch.tensor([0, 1, 250, 500, 998, 999])
    v = s.get_velocity(x0, nz, t)
    a = s.alphas_cumprod[t].double()[:, None, None]
    assert rel(v, a.sqrt() * nz.double() - (1 - a).sqrt() * x0.double()) < 1e-6
    assert torch.equal(v, po.velocity(x0, nz, t))
    # epsilon, x0 and v of one noisy sample describe the same point: x_t = sqrt(a) x0 + sqrt(1 - a) eps, v = sqrt(a) eps - sqrt(1 - a) x0
    xt = s.add_noise(x0, nz, t)
    assert rel(a.sqrt() * xt.double() - (1 - a).sqrt() * v.double(), x0.double()) < 1e-6


def test_compute_snr_and_min_snr_weights():
    import prediction_oracle as po
    s = DDPMScheduler()
    t = torch.tensor([0, 1, 100, 500, 900, 999])
    snr = compute_snr(s, t)
    a = s.alphas_cumprod[t].double()
    assert rel(snr, a / (1 - a)) < 1e-6 and snr.dtype == torch.float32
    assert snr[0] > 5e3 and snr[-1] < 1e-4                      # the linear schedule spans about 8 decades
    for pt, want in [("epsilon", torch.clamp(snr, max=5.0) / snr), ("v_prediction", torch.clamp(snr, max=5.0) / (snr + 1)),
                     ("sample", torch.clamp(snr, max=5.0))]:
        w = po.min_snr_weights(t, 5.0, pt)
        assert torch.equal(w, want), pt


def _gaussian_loop(sched, n, pt, N=100_000, mu=0.0, s=0.577, **step_kw):
    """x0 ~ N(mu, s^2): E[eps | x_t] = sqrt(1 - a) (x_t - sqrt(a) mu) / (a s^2 + 1 - a), and the exact x0 / v predictors follow from
    it (test_schedulers_host.py's target), in float64 with seeded noise for the stochastic steps."""
    sched.set_timesteps(n)
    acp = sched.alphas_cumprod.double()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(N, generator=g, dtype=torch.float64)
    for t in sched.timesteps.tolist():
        a = acp[t]
        eps = (1 - a).sqrt() * (x - a.sqrt() * mu) / (a * s * s + 1 - a)
        x0 = (x - (1 - a).sqrt() * eps) / a.sqrt()
        out = {"epsilon": eps, "sample": x0, "v_prediction": a.sqrt() * eps - (1 - a).sqrt() * x0}[pt]
        nz = torch.randn(N, generator=g, dtype=torch.float64)
        if isinstance(sched, DDPMScheduler):
            x = sched.step(out, t, x, noise=nz)
        elif isinstance(sched, DDIMScheduler):
            x = sched.step(out, t, x, variance_noise=nz, **step_kw).prev_sample
        else:
            x = sched.step(out, t, x).prev_sample
    return x


@pytest.mark.parametrize("kind,n,kw", [("ddpm", 100, {}), ("ddim", 50, {"eta": 0.0}), ("ddim", 50, {"eta": 1.0}), ("dpm", 20, {}),
                                       ("dpm", 200, {})])
def test_gaussian_target_loops_agree_across_parameterisations(kind, n, kw):
    """With exact predictors the three loops take the same path.  The loops run in float64, but the schedulers' coefficients
    (sqrt(a), sqrt(1 - a)) are fp32 0-d tensors, as in diffusers: each parameterisation's conversion carries their ~6e-8 relative
    rounding, hence 1e-6 rather than float64 agreement.  The samples keep the target's scale."""
    res = {pt: _gaussian_loop(_scheds(pt)[kind], n, pt, **kw) for pt in PRED_TYPES}
    for pt in ("sample", "v_prediction"):
        assert rel(res[pt], res["epsilon"]) <= 1e-6, (kind, n, pt, rel(res[pt], res["epsilon"]))
    assert 0.4 < res["epsilon"].std().item() < 0.8
