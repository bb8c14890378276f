"""CPU: the few-step samplers (DDIMSampler, DPMSolverSampler) -- their timestep schedules against the oracle's restatement of
diffusers 0.15 DDIMScheduler / DPMSolverMultistepScheduler, argument checks in Python and at the C ABI (no launch) -- and the
restatements themselves: per-step identities between the schedulers, and convergence of both loops to the exact answer for a
Gaussian target whose epsilon-predictor is known in closed form."""
import os
import sys

import pytest
import torch

from util import ROOT, load_cfg, rel

sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))
from diffusers import DDPMScheduler  # noqa: E402
from diffusers.schedulers_few_step import DDIMScheduler, DPMSolverMultistepScheduler  # noqa: E402


@pytest.fixture(scope="module")
def cpu_model():
    from prompt_tts_b200.models import TTSSingleSpeaker
    return TTSSingleSpeaker(load_cfg("tiny"))


@pytest.mark.parametrize("n", [1, 5, 20, 25, 50, 100, 333, "max"])
def test_sampler_timesteps_match_the_schedulers(cpu_model, n):
    from prompt_tts_b200.sample import DDIMSampler, DPMSolverSampler
    n_ddim, n_dpm = (1000, 999) if n == "max" else (n, n)
    ddim, dpm = DDIMScheduler(), DPMSolverMultistepScheduler()
    ddim.set_timesteps(n_ddim)
    dpm.set_timesteps(n_dpm)
    assert DDIMSampler(cpu_model, n_infer=n_ddim).timesteps == ddim.timesteps.tolist()
    assert DPMSolverSampler(cpu_model, n_infer=n_dpm).timesteps == dpm.timesteps.tolist()


def test_dpm_solver_grid():
    s = DPMSolverMultistepScheduler()
    s.set_timesteps(20)
    # k * 999 / 20 rounded half to even: 499.5 -> 500
    assert s.timesteps.tolist() == [999, 949, 899, 849, 799, 749, 699, 649, 599, 549, 500, 450, 400, 350, 300, 250, 200, 150, 100, 50]
    s.set_timesteps(1000)                     # the rounded grid repeats 500 (h = 0): why DPMSolverSampler stops at 999
    assert len(set(s.timesteps.tolist())) == 999


@pytest.mark.parametrize("n", [10, 20, 50])
def test_ddim_eta_one_is_the_ddpm_step(n):
    """DDIM with eta = 1 is the DDPM ancestral step (no clipping on either side, same noise).  Both evaluate 1 - a_t / a_prev in
    fp32, which loses digits as the step shrinks near t = 0: 3.3e-6 apart at (20 -> 0), 1.3e-5 at (10 -> 0)."""
    g = torch.Generator().manual_seed(n)
    ddim, ddpm = DDIMScheduler(clip_sample=False), DDPMScheduler(clip_sample=False)
    ddim.set_timesteps(n)
    ddpm.set_timesteps(n)
    for t in ddim.timesteps.tolist()[:: max(1, n // 5)] + [int(ddim.timesteps[-2]), 0]:
        x, eps, nz = (torch.randn(4, 8, 64, generator=g) for _ in range(3))
        a = ddim.step(eps, t, x, eta=1.0, variance_noise=nz).prev_sample
        b = ddpm.step(eps, t, x, noise=nz)
        assert rel(a, b) <= 1e-5, (n, t, rel(a, b))


@pytest.mark.parametrize("t", [980, 500, 100, 20])
def test_dpm_first_order_is_deterministic_ddim(t):
    """The first-order DPM-Solver++ update from t to t - 20 equals DDIM (eta = 0, no clipping) over the same pair."""
    g = torch.Generator().manual_seed(t)
    ddim, dpm = DDIMScheduler(clip_sample=False), DPMSolverMultistepScheduler()
    ddim.set_timesteps(50)
    x, eps = (torch.randn(4, 8, 64, generator=g) for _ in range(2))
    a = ddim.step(eps, t, x, eta=0.0).prev_sample
    b = dpm.dpm_solver_first_order_update(dpm.convert_model_output(eps, t, x), t, t - 20, x)
    assert rel(b, a) <= 1e-5, rel(b, a)


def test_dpm_second_order_with_equal_predictions_is_first_order():
    g = torch.Generator().manual_seed(1)
    dpm = DPMSolverMultistepScheduler()
    x, m = (torch.randn(4, 8, 64, generator=g) for _ in range(2))
    for s1, s0, t in [(999, 949, 899), (600, 550, 500), (100, 50, 0)]:
        one = dpm.dpm_solver_first_order_update(m, s0, t, x)
        two = dpm.multistep_dpm_solver_second_order_update([m, m], [s1, s0], t, x)
        assert torch.equal(one, two)


def _gaussian_loop(sched, n, N=100_000, mu=0.0, s=0.577, **step_kw):
    """x0 ~ N(mu, s^2): x_t ~ N(sqrt(a) mu, a s^2 + 1 - a) and E[eps | x_t] = sqrt(1 - a) (x_t - sqrt(a) mu) / (a s^2 + 1 - a)."""
    sched.set_timesteps(n)
    acp = sched.alphas_cumprod.double()
    x = torch.randn(N, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    for t in sched.timesteps.tolist():
        a = acp[t]
        eps = (1 - a).sqrt() * (x - a.sqrt() * mu) / (a * s * s + 1 - a)
        x = sched.step(eps, t, x, **step_kw).prev_sample
    return x


def test_schedulers_converge_on_a_gaussian_target():
    """With the exact predictor both loops approach N(0, 0.577^2) as steps grow (1e5 samples: ~0.2 % sampling noise on the
    std).  Few-step quality is not asserted: at 20 steps on this schedule DPM-Solver++'s second-order last step overshoots
    the std by ~20 %."""
    s = 0.577
    for sched, n, kw in [(DPMSolverMultistepScheduler(), 200, {}), (DPMSolverMultistepScheduler(), 500, {}),
                         (DDIMScheduler(clip_sample=False), 1000, {"eta": 0.0})]:
        x = _gaussian_loop(sched, n, s=s, **kw)
        assert abs(x.std().item() / s - 1) < 0.01 and abs(x.mean().item()) < 0.01, (type(sched).__name__, n, x.std().item())


def test_fast_samplers_check_their_arguments(cpu_model):
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.sample import DDIMSampler, DPMSolverSampler
    for bad in (0, 1001, 2.5):
        with pytest.raises(ValueError):
            DDIMSampler(cpu_model, n_infer=bad)
    for bad in (0, 1000):
        with pytest.raises(ValueError):
            DPMSolverSampler(cpu_model, n_infer=bad)
    for eta in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            DDIMSampler(cpu_model, eta=eta)
    assert DDIMSampler(cpu_model).n_infer == 50 and DPMSolverSampler(cpu_model).n_infer == 20
    for smp in (DDIMSampler(cpu_model, n_infer=2, eta=1.0), DPMSolverSampler(cpu_model, n_infer=2)):
        with pytest.raises(_lib.PtError):                  # CPU tensors: there is no CPU fallback
            smp.sample(torch.zeros(1, 24, dtype=torch.int32), 16)


def test_ddpm_sampler_checks_n_infer(cpu_model):
    """n_infer = 0 would divide by zero and n_infer > n_train would give a zero stride (every timestep 0)"""
    from prompt_tts_b200.sample import DDPMSampler
    for bad, n_train in ((0, 1000), (1001, 1000), (11, 10), (True, 1000), (2.5, 1000), ("5", 1000)):
        with pytest.raises(ValueError, match="n_infer"):
            DDPMSampler(cpu_model, n_infer=bad, n_train=n_train)
    assert DDPMSampler(cpu_model).n_infer == 100 and DDPMSampler(cpu_model, n_infer=10, n_train=10).stride == 1
    assert DDPMSampler(cpu_model, n_infer=5.0).timesteps == [800, 600, 400, 200, 0]


def test_step_entry_points_validate_their_scalars():
    """pt_ddim_step / pt_dpmpp_step refuse bad scalars before anything is launched (no device needed).  Pointers are never
    dereferenced on these paths: each call fails validation first."""
    from prompt_tts_b200 import _lib, ops
    buf = torch.zeros(64)
    p, z = ops._p(buf), ops._p(None)

    def ddim(*, noise=p, prompt=z, keep=0, n=64, T=16, acp_t=0.5, acp_prev=0.6, eta=0.0, pa=1.0, pb=0.0):
        ops.call("ddim_step", p, p, noise, prompt, z, p, n, T, keep, acp_t, acp_prev, eta, pa, pb, z)

    def dpmpp(*, m_prev=p, order=2, keep=0, n=64, T=16, s0=0.5, s1=0.4, t=0.6):
        ops.call("dpmpp_step", p, p, m_prev, p, z, z, p, n, T, keep, s0, s1, t, order, 1.0, 0.0, z)

    cases = [(lambda: ddim(acp_t=0.0), "acp_t"), (lambda: ddim(acp_prev=0.4), "acp_prev"), (lambda: ddim(acp_prev=1.5), "acp_prev"),
             (lambda: ddim(eta=-1.0), "eta"), (lambda: ddim(eta=1.0, noise=z), "noise required"), (lambda: ddim(eta=5.0), "too large"),
             (lambda: ddim(n=60), "n=60"), (lambda: ddim(keep=17), "keep=17"), (lambda: ddim(keep=4), "in-painting"),
             (lambda: dpmpp(order=3), "order=3"), (lambda: dpmpp(m_prev=z), "order=2"), (lambda: dpmpp(t=0.5), "acp_t"),
             (lambda: dpmpp(s1=0.5), "acp_s1"), (lambda: dpmpp(s0=1.0, t=1.0), "acp_s0")]
    for fn, msg in cases:
        with pytest.raises(_lib.PtError, match=msg):
            fn()
