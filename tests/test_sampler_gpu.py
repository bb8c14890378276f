"""GPU: the DDPM sampling step kernel and the 100-step sampler loop (SURVEY 8 row N1) against the oracle's restatement of
diffusers 0.15 `DDPMScheduler.step` / the reference denoiser (oracle/ref_model.py), on identical seeded inputs."""
import pytest
import torch

import sampling_oracle as so
from util import load_model, rel, synth_inputs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("t", [990, 500, 10, 0])
def test_ddpm_step_matches_oracle(cuda, t):
    import ref_model
    from prompt_tts_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(t)
    x = torch.randn(3, 8, 40, device=cuda, generator=g)
    eps = torch.randn(3, 8, 40, device=cuda, generator=g)
    nz = torch.randn(3, 8, 40, device=cuda, generator=g)
    acp = ref_model.ddpm_alphas_cumprod()
    out = torch.empty_like(x)
    acp_prev = float(acp[t - 10]) if t >= 10 else 1.0
    ops.call("ddpm_step", ops._p(eps), ops._p(x), ops._p(nz if t >= 10 else None), ops._p(None), ops._p(out), x.numel(), 40, 0,
             float(acp[t]), acp_prev, ops._stream())
    ref = ref_model.ddpm_step(eps.cpu(), t, x.cpu(), nz.cpu())
    assert rel(out.cpu(), ref) < 2e-6


def test_sampler_matches_oracle_loop(cuda):
    from prompt_tts_b200.sample import DDPMSampler
    cfg, model = load_model("tiny", cuda)
    B, T, n_infer = 2, 16, 5
    inp = synth_inputs(cfg, B, T, seed=5, device=cuda)
    g = torch.Generator(device="cuda").manual_seed(9)
    x_T = torch.randn(B, cfg["in_channels"], T, device=cuda, generator=g)
    noises = torch.randn(n_infer, B, cfg["in_channels"], T, device=cuda, generator=g)
    outs = {}
    for graph in (False, True):
        outs[graph] = DDPMSampler(model, n_infer=n_infer, use_graph=graph).sample(inp["ids"], T, x_T=x_T, noises=noises)
    # GroupNorm statistics are accumulated with fp32 atomics (order not fixed), so two runs agree to rounding, not bit for bit
    assert rel(outs[False], outs[True]) < 1e-3, "graph replay must reproduce the eager loop"
    # oracle loop: fp32 reference modules + DDPMScheduler.step restatement, same x_T / noises
    x = so.oracle_loop(model, cfg, "ddpm", None, n_infer, inp["ids"], x_T, noises)
    e = rel(outs[True], x)
    print(f"\n[sampler tiny, {n_infer} steps] rel err vs fp32 oracle loop {e:.2e}")
    assert e < 2e-2 * 2, e          # bf16 denoiser error (<= 2e-2 per call) compounds over the steps; the scheduler step itself is exact


def test_sampler_prompt_inpainting_and_codes(cuda):
    from prompt_tts_b200.sample import DDPMSampler
    cfg, model = load_model("tiny", cuda)
    B, T, P = 2, 16, 6
    inp = synth_inputs(cfg, B, T, seed=6, device=cuda)
    prompt = inp["x0"][..., :P].contiguous()
    smp = DDPMSampler(model, n_infer=4)
    x = smp.sample(inp["ids"], T, prompt=prompt, seed=3)
    assert torch.equal(x[..., :P], prompt), "the prompt frames must come out clean"
    assert torch.isfinite(x).all() and x.abs().max() <= 1.0 + 1e-6      # clip_sample
    codes = smp.sample(inp["ids"], T, prompt=prompt, seed=3, return_codes=True)
    ref = torch.clamp(torch.round((x + 1) * 511.5), 0, 1023).to(torch.int64)
    assert torch.equal(codes, ref)
    assert torch.equal(codes[..., :P], torch.round((prompt + 1) * 511.5).to(torch.int64))     # prompt codes round-trip exactly


def test_sampler_prompt_tokens_extend_the_cross_attention_context(cuda):
    """Optional speech-prompt tokens appended to the text encoding (SURVEY 8 row N2 hook, default off): the run with tokens equals
    the oracle loop whose encoder_hidden_states is [text encoding | tokens], and differs from the run without them."""
    from prompt_tts_b200.sample import DDPMSampler
    cfg, model = load_model("tiny", cuda)
    B, T, n_infer, P = 2, 16, 3, 9
    inp = synth_inputs(cfg, B, T, seed=8, device=cuda)
    g = torch.Generator(device="cuda").manual_seed(4)
    x_T = torch.randn(B, cfg["in_channels"], T, device=cuda, generator=g)
    noises = torch.randn(n_infer, B, cfg["in_channels"], T, device=cuda, generator=g)
    toks = torch.randn(B, P, cfg["cross_attention_dim"], device=cuda, generator=g)
    smp = DDPMSampler(model, n_infer=n_infer)
    with_t = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, prompt_tokens=toks)
    without = smp.sample(inp["ids"], T, x_T=x_T, noises=noises)
    assert rel(with_t, without) > 1e-3
    x = so.oracle_loop(model, cfg, "ddpm", None, n_infer, inp["ids"], x_T, noises, toks=toks)
    assert rel(with_t, x) < 4e-2
