"""The sampler tests' shared oracle: the product's three samplers built by kind, and one fp32 loop of oracle/ref_model.py's denoiser
and the oracle schedulers of tests/prediction_oracle.py (whose epsilon paths are the shim's) on the same seeded inputs."""
import torch

import prediction_oracle as po
from util import rel, synth_inputs


def make_sampler(model, kind, eta, n_infer, pt="epsilon", use_graph=True):
    """kind "ddpm", "ddim" (eta) or "dpm" """
    from prompt_tts_b200.sample import DDIMSampler, DDPMSampler, DPMSolverSampler
    if kind == "ddpm":
        return DDPMSampler(model, n_infer=n_infer, use_graph=use_graph, prediction_type=pt)
    if kind == "ddim":
        return DDIMSampler(model, n_infer=n_infer, eta=eta, use_graph=use_graph, prediction_type=pt)
    return DPMSolverSampler(model, n_infer=n_infer, use_graph=use_graph, prediction_type=pt)


def case(cfg, B, T, n_infer, seed, dev):
    """a synthetic batch, x_T and the per-step noises"""
    inp = synth_inputs(cfg, B, T, seed=seed, device=dev)
    g = torch.Generator(device="cuda").manual_seed(seed + 100)
    x_T = torch.randn(B, cfg["in_channels"], T, device=dev, generator=g)
    noises = torch.randn(n_infer, B, cfg["in_channels"], T, device=dev, generator=g)
    return inp, x_T, noises


def oracle_loop(model, cfg, kind, eta, n_infer, ids, x_T, noises, pt="epsilon", w=None, prompt=None, prompt_noise=None, toks=None,
                eps_err=0.0, err_seed=None):
    """fp32 loop: ref_model.text_encoder once (toks appended to its output as extra tokens), ref_model.unet, the oracle scheduler's
    step for a model output of type pt; prompt frames overwritten after every step with the prompt noised to the level the step
    landed on (clean after the last step).  w None: the conditional output alone.  w a number: also ref_model.unet on a zero context
    and the guided output u + w (c - u), formed even at w = 1.  eps_err > 0 adds a Gaussian error of that relative size to every
    denoiser output, drawn from a generator seeded with err_seed (each test file keeps its own): what the loop itself makes of a
    given per-call error."""
    import ref_model
    acp = ref_model.ddpm_alphas_cumprod().to(x_T.device)
    if kind == "ddpm":
        ts = [k * (1000 // n_infer) for k in range(n_infer)][::-1]
    else:
        sched = po.DDIMScheduler(prediction_type=pt) if kind == "ddim" else po.DPMSolverMultistepScheduler(prediction_type=pt)
        sched.set_timesteps(n_infer)
        ts = sched.timesteps.tolist()
    sd = {k: v.detach().float() for k, v in model.state_dict().items()}
    B = x_T.shape[0]
    g = torch.Generator(device=x_T.device).manual_seed(err_seed) if eps_err > 0 else None

    def err(e):
        return e + eps_err * e.norm() / e.numel() ** 0.5 * torch.randn(e.shape, device=e.device, generator=g) if eps_err > 0 else e

    with torch.no_grad():
        enc = ref_model.text_encoder(sd, cfg, ids)
        if toks is not None:
            enc = torch.cat([enc, toks], dim=1)
        x = x_T.clone()
        for i, t in enumerate(ts):
            tt = torch.full((B,), t, device=x.device, dtype=torch.int64)
            o = err(ref_model.unet(sd, cfg, x, tt, enc))
            if w is not None:
                u = err(ref_model.unet(sd, cfg, x, tt, torch.zeros_like(enc)))
                o = u + w * (o - u)
            if kind == "ddpm":
                x = po.ddpm_step(o, t, x, noises[i], acp=acp, n_infer=n_infer, prediction_type=pt)
                to = t - 1000 // n_infer
            elif kind == "ddim":
                x = sched.step(o, t, x, eta=eta, variance_noise=noises[i]).prev_sample
                to = t - 1000 // n_infer
            else:
                x = sched.step(o, t, x).prev_sample
                to = ts[i + 1] if i + 1 < n_infer else -1
            if prompt is not None:
                keep = prompt.shape[-1]
                if i == n_infer - 1 or to < 0:
                    x[..., :keep] = prompt
                else:
                    x[..., :keep] = acp[to].sqrt() * prompt + (1 - acp[to]).sqrt() * prompt_noise[i]
    return x


def grad_err(model, ref_grads):
    """relative error of the model's global gradient vector over the parameters the oracle's autograd reached (an oracle gradient
    that is None or all zero, as the dead proj_out weights' is, is skipped)"""
    named = dict(model.named_parameters())
    keys = sorted(k for k, g in ref_grads.items() if g is not None and g.abs().max() > 0)
    assert all(named[k].grad is not None for k in keys), [k for k in keys if named[k].grad is None][:5]
    return rel(torch.cat([named[k].grad.flatten() for k in keys]), torch.cat([ref_grads[k].flatten() for k in keys]))
