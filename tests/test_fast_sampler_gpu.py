"""GPU: the few-step sampling kernels (pt_ddim_step, pt_dpmpp_step) against the oracle's restatement of diffusers 0.15
DDIMScheduler / DPMSolverMultistepScheduler, and DDIMSampler / DPMSolverSampler end to end against an fp32 oracle loop (shim
scheduler + oracle/ref_model.py denoiser) on identical seeded inputs."""
import os
import sys

import pytest
import torch

import sampling_oracle as so
from util import ROOT, load_model, rel, synth_inputs

sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))
from diffusers.schedulers_few_step import DDIMScheduler, DPMSolverMultistepScheduler  # noqa: E402

pytestmark = pytest.mark.gpu

SHAPE = (3, 8, 40)


@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("t", [990, 500, 10, 0])
def test_ddim_step_matches_scheduler(cuda, t, eta):
    from prompt_tts_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(t)
    x, eps, nz = (torch.randn(*SHAPE, device=cuda, generator=g) for _ in range(3))
    sched = DDIMScheduler()
    sched.set_timesteps(100)
    acp = sched.alphas_cumprod
    out = torch.empty_like(x)
    ops.call("ddim_step", ops._p(eps), ops._p(x), ops._p(nz if eta > 0 else None), ops._p(None), ops._p(None), ops._p(out), x.numel(),
             SHAPE[-1], 0, float(acp[t]), float(acp[t - 10]) if t >= 10 else 1.0, eta, 1.0, 0.0, ops._stream())
    ref = sched.step(eps.cpu(), t, x.cpu(), eta=eta, variance_noise=nz.cpu()).prev_sample
    assert rel(out.cpu(), ref) < 2e-6


def _dpm_case(n, k, seed):
    """Drive the shim through steps 0..k-1 with a plausible model (x_t from a fixed x0, eps = the true noise + 10 % error) and
    return the inputs of step k and the shim's result: (x, eps, previous x0 prediction, order, acp triple, prev_sample, m0)."""
    sched = DPMSolverMultistepScheduler()
    sched.set_timesteps(n)
    ts, acp = sched.timesteps.tolist(), sched.alphas_cumprod
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(*SHAPE, generator=g) * 2 - 1
    for j in range(k + 1):
        a = acp[ts[j]]
        nz = torch.randn(*SHAPE, generator=g)
        x = a.sqrt() * x0 + (1 - a).sqrt() * nz
        eps = nz + 0.1 * torch.randn(*SHAPE, generator=g)
        m_prev = sched.model_outputs[-1]
        out = sched.step(eps, ts[j], x).prev_sample
    last = k == n - 1
    order = 1 if k == 0 or (last and n < 15) else 2
    acps = (float(acp[ts[k]]), float(acp[ts[k - 1]]) if order == 2 else 0.0, float(acp[0 if last else ts[k + 1]]))
    return x, eps, m_prev, order, acps, out, sched.model_outputs[-1]


@pytest.mark.parametrize("n,k", [(20, 0), (20, 1), (20, 10), (20, 19), (5, 4)])
def test_dpmpp_step_matches_scheduler(cuda, n, k):
    """first step (order 1), second step, a middle one and the last (order 2 at 20 steps; order 1 below 15 steps)"""
    from prompt_tts_b200 import ops
    x, eps, m_prev, order, (a0, a1, at), ref, ref_m = _dpm_case(n, k, 100 * n + k)
    x, eps = x.to(cuda), eps.to(cuda)
    hist = m_prev.to(cuda) if m_prev is not None else torch.full_like(x, float("nan"))    # order 1 must not read it
    out = torch.empty_like(x)
    ops.call("dpmpp_step", ops._p(eps), ops._p(x), ops._p(hist), ops._p(hist), ops._p(None), ops._p(None), ops._p(out), x.numel(),
             SHAPE[-1], 0, a0, a1, at, order, 1.0, 0.0, ops._stream())
    assert (order == 2) == (k > 0 and not (k == n - 1 and n < 15))
    assert rel(out.cpu(), ref) < 2e-6, rel(out.cpu(), ref)
    assert rel(hist.cpu(), ref_m) < 2e-6, "the history buffer must hold this step's x0 prediction"


def test_step_kernels_inpaint_prompt_frames(cuda):
    """keep > 0: the first `keep` frames of every row are p_a * prompt + p_b * prompt_noise, every other frame is the step's own
    result bit for bit, and the DPM-Solver history keeps the model's prediction in the prompt frames too."""
    from prompt_tts_b200 import ops
    B, C, T = SHAPE
    keep = 7
    g = torch.Generator(device="cuda").manual_seed(2)
    prompt, pn = torch.rand(B, C, keep, device=cuda, generator=g) * 2 - 1, torch.randn(B, C, keep, device=cuda, generator=g)
    x, eps, nz, m1 = (torch.randn(*SHAPE, device=cuda, generator=g) for _ in range(4))
    pa, pb = 0.8, 0.6
    want = pa * prompt + pb * pn
    acp = DDIMScheduler().alphas_cumprod
    for kind in ("ddim", "dpmpp"):
        outs, hists = [], []
        for k, pp, pq in ((0, None, None), (keep, prompt, pn)):
            out, hist = torch.empty_like(x), m1.clone()
            if kind == "ddim":
                ops.call("ddim_step", ops._p(eps), ops._p(x), ops._p(nz), ops._p(pp), ops._p(pq), ops._p(out), x.numel(), T, k,
                         float(acp[500]), float(acp[480]), 1.0, pa, pb, ops._stream())
            else:
                ops.call("dpmpp_step", ops._p(eps), ops._p(x), ops._p(hist), ops._p(hist), ops._p(pp), ops._p(pq), ops._p(out), x.numel(),
                         T, k, float(acp[500]), float(acp[550]), float(acp[450]), 2, pa, pb, ops._stream())
            outs.append(out)
            hists.append(hist)
        assert torch.equal(outs[1][..., keep:], outs[0][..., keep:]), kind
        assert rel(outs[1][..., :keep], want) < 1e-6, kind
        assert torch.equal(hists[1], hists[0]), kind
    # clean prompt: p_a = 1, p_b = 0 copies it exactly and never reads the (absent) noise
    out = torch.empty_like(x)
    ops.call("ddim_step", ops._p(eps), ops._p(x), ops._p(None), ops._p(prompt), ops._p(None), ops._p(out), x.numel(), T, keep,
             float(acp[10]), 1.0, 0.0, 1.0, 0.0, ops._stream())
    assert torch.equal(out[..., :keep], prompt)


# ---------------------------------------------------------------------------------------------------------- whole loop
SAMPLERS = [("ddim", 0.0), ("ddim", 1.0), ("dpm", None)]


@pytest.fixture(scope="module")
def tiny(cuda):
    return load_model("tiny", cuda)


@pytest.mark.parametrize("kind,eta", SAMPLERS)
def test_fast_sampler_matches_oracle_loop(cuda, tiny, kind, eta):
    cfg, model = tiny
    B, T, n_infer = 2, 16, 5
    inp = synth_inputs(cfg, B, T, seed=5, device=cuda)
    g = torch.Generator(device="cuda").manual_seed(9)
    x_T = torch.randn(B, cfg["in_channels"], T, device=cuda, generator=g)
    noises = torch.randn(n_infer, B, cfg["in_channels"], T, device=cuda, generator=g)
    outs = {graph: so.make_sampler(model, kind, eta, n_infer, use_graph=graph).sample(inp["ids"], T, x_T=x_T, noises=noises)
            for graph in (False, True)}
    # GroupNorm statistics are accumulated with fp32 atomics (order not fixed), so two runs agree to rounding, not bit for bit
    assert rel(outs[False], outs[True]) < 1e-3, "graph replay must reproduce the eager loop"
    x = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises)
    e = rel(outs[True], x)
    bound = 2e-2 * 2                # bf16 denoiser error (<= 2e-2 per call) carried through the steps; the step kernels are exact
    if kind == "ddim" and eta == 0.0:
        # Deterministic DDIM with clipping carries a denoiser error much further on this random-weight model: the error of an
        # early eps passes through x0 = (x - sqrt(1 - a_t) eps) / sqrt(a_t) and is scaled by sqrt(a_prev / a_t) at every later
        # step, and no fresh noise dilutes it.  The fp32 oracle loop alone turns a 1e-2 random per-call error into 8e-2 at the
        # output here (DDPM 0.7e-2, eta = 1 1.1e-2, DPM-Solver++ 0.35e-2); the product (6.2e-2) is held to what the oracle loop
        # makes of the per-call bar of 2e-2.
        bound = rel(so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, eps_err=2e-2, err_seed=17), x)
    print(f"\n[{kind} eta={eta} tiny, {n_infer} steps] rel err vs fp32 oracle loop {e:.2e} (bound {bound:.2e})")
    assert e < bound, (e, bound)


@pytest.mark.parametrize("kind,eta", SAMPLERS)
def test_fast_sampler_prompt_inpainting_and_codes(cuda, tiny, kind, eta):
    cfg, model = tiny
    B, T, P, n_infer = 2, 16, 6, 4
    inp = synth_inputs(cfg, B, T, seed=6, device=cuda)
    prompt = inp["x0"][..., :P].contiguous()
    smp = so.make_sampler(model, kind, eta, n_infer)
    x = smp.sample(inp["ids"], T, prompt=prompt, seed=3)
    assert torch.equal(x[..., :P], prompt), "the prompt frames must come out clean"
    assert torch.isfinite(x).all()
    codes = smp.sample(inp["ids"], T, prompt=prompt, seed=3, return_codes=True)
    ref = torch.clamp(torch.round((x + 1) * 511.5), 0, 1023).to(torch.int64)
    assert torch.equal(codes, ref)
    assert torch.equal(codes[..., :P], torch.round((prompt + 1) * 511.5).to(torch.int64))     # prompt codes round-trip exactly
    # the same run with explicit noises against the oracle loop that overwrites the prompt frames after every step
    g = torch.Generator(device="cuda").manual_seed(11)
    x_T = torch.randn(B, cfg["in_channels"], T, device=cuda, generator=g)
    noises = torch.randn(n_infer, B, cfg["in_channels"], T, device=cuda, generator=g)
    pn = torch.randn(n_infer, B, cfg["in_channels"], P, device=cuda, generator=g)
    got = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, prompt=prompt, prompt_noise=pn)
    want = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, prompt=prompt, prompt_noise=pn)
    assert torch.equal(got[..., :P], want[..., :P])
    assert rel(got, want) < 4e-2, rel(got, want)
    with pytest.raises(Exception, match="prompt must be"):
        smp.sample(inp["ids"], T, prompt=prompt, prompt_noise=pn[:, :1])


@pytest.mark.parametrize("kind,eta", [("ddim", 0.0), ("dpm", None)])
def test_fast_sampler_prompt_tokens(cuda, tiny, kind, eta):
    """prompt tokens appended to the text encoding change the result, which equals the oracle loop conditioned on
    [text encoding | tokens]"""
    cfg, model = tiny
    B, T, n_infer, P = 2, 16, 3, 9
    inp = synth_inputs(cfg, B, T, seed=8, device=cuda)
    g = torch.Generator(device="cuda").manual_seed(4)
    x_T = torch.randn(B, cfg["in_channels"], T, device=cuda, generator=g)
    noises = torch.randn(n_infer, B, cfg["in_channels"], T, device=cuda, generator=g)
    toks = torch.randn(B, P, cfg["cross_attention_dim"], device=cuda, generator=g)
    smp = so.make_sampler(model, kind, eta, n_infer)
    with_t = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, prompt_tokens=toks)
    without = smp.sample(inp["ids"], T, x_T=x_T, noises=noises)
    assert rel(with_t, without) > 1e-3
    x = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, toks=toks)
    assert rel(with_t, x) < 4e-2, rel(with_t, x)
