"""GPU: sample / v prediction and Min-SNR-gamma weighting.  pt_diffusion_loss against torch (the v target bit for bit), the
`_pred` step entry points against the oracle's schedulers extended to these types (tests/prediction_oracle.py) and, for
epsilon, bit for bit against the entry points without the suffix; kernel-driven loops of the three exact predictors of a Gaussian target against each other; DenoiserTrainStep
against the oracle's fp32 autograd (eager and graph-replayed); the three samplers' loops against an fp32 oracle loop; launch
counts."""

import pytest
import torch

import prediction_oracle as po
import sampling_oracle as so
from prediction_oracle import DDIMScheduler, DDPMScheduler, DPMSolverMultistepScheduler
from util import rel, synth_inputs

pytestmark = pytest.mark.gpu
TOL = 2e-2
PRED = {"epsilon": 0, "sample": 1, "v_prediction": 2}
NON_EPS = ("sample", "v_prediction")
SHAPE = (3, 8, 40)


# ---------------------------------------------------------------------------------------------------------------- loss kernel
def _loss_case(dev, seed=0):
    from prompt_tts_b200.train import ddpm_tables
    B, C, T = 8, 8, 64                                  # n = 4096: 2 / n is a power of two, so dpred = -2 target / n exactly at pred = 0
    g = torch.Generator(device="cuda").manual_seed(seed)
    x0 = torch.rand(B, C, T, device=dev, generator=g) * 2 - 1
    noise = torch.randn(B, C, T, device=dev, generator=g)
    pred = torch.randn(B, C, T, device=dev, generator=g)
    t = torch.tensor([0, 999, 1, 500, 998, 250, 10, 700], dtype=torch.int64, device=dev)
    sa, sb = ddpm_tables(device=dev)
    return x0, noise, pred, t, sa, sb


def _diffusion_loss(pred, x0, noise, t, sa, sb, pt, gamma, gs):
    from prompt_tts_b200 import ops
    loss = torch.zeros((), device=pred.device)
    dpred = torch.full_like(pred, float("nan"))
    ops.call("diffusion_loss", ops._p(pred), ops._p(x0), ops._p(noise), ops._p(t), ops._p(sa), ops._p(sb), ops._p(loss), ops._p(dpred),
             pred.shape[0], pred[0].numel(), PRED[pt], gamma, gs, ops._stream())
    return loss, dpred


def _target(pt, x0, noise, t):
    return {"epsilon": noise, "sample": x0}.get(pt) if pt != "v_prediction" else po.velocity(x0, noise, t)


@pytest.mark.parametrize("pt", list(PRED))
def test_diffusion_loss_target_is_bitwise(cuda, pt):
    """with pred = 0, w = 1, gscale = 1: dpred = -2 target / n exactly, so the kernel's target is read back bit for bit"""
    x0, noise, _, t, sa, sb = _loss_case(cuda, 1)
    zero = torch.zeros_like(x0)
    _, dpred = _diffusion_loss(zero, x0, noise, t, sa, sb, pt, 0.0, 1.0)
    got = dpred * (-x0.numel() / 2)
    assert torch.equal(got, _target(pt, x0, noise, t))


@pytest.mark.parametrize("gs", [1.0, 1.5 / 4])             # gscale; gscale / accumulation_steps as the train step passes it
@pytest.mark.parametrize("gamma", [None, 5.0])
@pytest.mark.parametrize("pt", list(PRED))
def test_diffusion_loss_matches_torch(cuda, pt, gamma, gs):
    x0, noise, pred, t, sa, sb = _loss_case(cuda, 2)
    loss, dpred = _diffusion_loss(pred, x0, noise, t, sa, sb, pt, 0.0 if gamma is None else gamma, gs)
    target = _target(pt, x0, noise, t)
    w = torch.ones(8, device=cuda) if gamma is None else po.min_snr_weights(t, gamma, pt)
    d = pred - target
    want_loss = ((d * d).mean(dim=(1, 2)) * w).mean()
    want_dpred = 2 * w[:, None, None] * d / d.numel() * gs
    if gamma is not None:
        assert w.max() / w.min() > 10, "t = 0 and t = 999 must be weighted differently"
    print(f"\n[diffusion_loss {pt} gamma={gamma} gscale={gs}] loss rel {rel(loss, want_loss):.1e} dpred rel {rel(dpred, want_dpred):.1e}")
    assert rel(loss, want_loss) < 1e-6 and rel(dpred, want_dpred) < 1e-6
    # the loss accumulates into its buffer, as pt_mse_fwd_bwd's does
    from prompt_tts_b200 import ops
    ops.call("diffusion_loss", ops._p(pred), ops._p(x0), ops._p(noise), ops._p(t), ops._p(sa), ops._p(sb), ops._p(loss), ops._p(dpred),
             8, pred[0].numel(), PRED[pt], 0.0 if gamma is None else gamma, gs, ops._stream())
    assert rel(loss, 2 * want_loss) < 1e-6


def test_diffusion_loss_epsilon_unweighted_is_mse(cuda):
    from prompt_tts_b200 import ops
    x0, noise, pred, t, sa, sb = _loss_case(cuda, 3)
    loss, dpred = _diffusion_loss(pred, x0, noise, t, sa, sb, "epsilon", 0.0, 0.5)
    l2, d2 = torch.zeros((), device=cuda), torch.empty_like(pred)
    ops.call("mse_fwd_bwd", ops._p(pred), ops._p(noise), ops._p(l2), ops._p(d2), pred.numel(), 0.5, ops._stream())
    assert torch.equal(dpred, d2) and rel(loss, l2) < 1e-6


# ---------------------------------------------------------------------------------------------------------------- step kernels
def _ddpm_call(name_pt, out_, x, nz, known, out, keep, a, ap):
    from prompt_tts_b200 import ops
    args = [ops._p(out_), ops._p(x), ops._p(nz), ops._p(known), ops._p(out), x.numel(), x.shape[-1], keep, a, ap]
    if name_pt is None:
        ops.call("ddpm_step", *args, ops._stream())
    else:
        ops.call("ddpm_step_pred", *args, PRED[name_pt], ops._stream())


def _ddim_call(name_pt, out_, x, nz, prompt, pn, out, keep, a, ap, eta, pa=1.0, pb=0.0):
    from prompt_tts_b200 import ops
    args = [ops._p(out_), ops._p(x), ops._p(nz), ops._p(prompt), ops._p(pn), ops._p(out), x.numel(), x.shape[-1], keep, a, ap, eta, pa, pb]
    if name_pt is None:
        ops.call("ddim_step", *args, ops._stream())
    else:
        ops.call("ddim_step_pred", *args, PRED[name_pt], ops._stream())


def _dpm_call(name_pt, out_, x, m_prev, m_out, prompt, pn, out, keep, a0, a1, at, order, pa=1.0, pb=0.0):
    from prompt_tts_b200 import ops
    args = [ops._p(out_), ops._p(x), ops._p(m_prev), ops._p(m_out), ops._p(prompt), ops._p(pn), ops._p(out), x.numel(), x.shape[-1], keep,
            a0, a1, at, order, pa, pb]
    if name_pt is None:
        ops.call("dpmpp_step", *args, ops._stream())
    else:
        ops.call("dpmpp_step_pred", *args, PRED[name_pt], ops._stream())


def _output(pt, x, a, g):
    """a plausible model output of type pt at (x, a): a random x0 in [-1.2, 1.2] (some of it clipped) and the eps it implies"""
    x0 = torch.rand(x.shape, device=x.device, generator=g) * 2.4 - 1.2
    if pt == "sample":
        return x0
    eps = (x - a.sqrt() * x0) / (1 - a).sqrt()
    return eps if pt == "epsilon" else a.sqrt() * eps - (1 - a).sqrt() * x0


@pytest.mark.parametrize("pt", NON_EPS)
@pytest.mark.parametrize("t", [990, 500, 10, 0])
def test_ddpm_step_pred_matches_scheduler(cuda, pt, t):
    g = torch.Generator(device="cuda").manual_seed(t + 7)
    x, nz = (torch.randn(*SHAPE, device=cuda, generator=g) for _ in range(2))
    sched = DDPMScheduler(prediction_type=pt)
    sched.set_timesteps(100)
    acp = sched.alphas_cumprod
    o = _output(pt, x, acp[t].to(cuda), g)
    out = torch.empty_like(x)
    _ddpm_call(pt, o, x, nz if t >= 10 else None, None, out, 0, float(acp[t]), float(acp[t - 10]) if t >= 10 else 1.0)
    ref = sched.step(o.cpu(), t, x.cpu(), noise=nz.cpu())
    assert rel(out.cpu(), ref) < 2e-6, rel(out.cpu(), ref)


@pytest.mark.parametrize("pt", NON_EPS)
@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("t", [990, 500, 10, 0])
def test_ddim_step_pred_matches_scheduler(cuda, pt, t, eta):
    g = torch.Generator(device="cuda").manual_seed(t + 11)
    x, nz = (torch.randn(*SHAPE, device=cuda, generator=g) for _ in range(2))
    sched = DDIMScheduler(prediction_type=pt)
    sched.set_timesteps(100)
    acp = sched.alphas_cumprod
    o = _output(pt, x, acp[t].to(cuda), g)
    out = torch.empty_like(x)
    _ddim_call(pt, o, x, nz if eta > 0 else None, None, None, out, 0, float(acp[t]), float(acp[t - 10]) if t >= 10 else 1.0, eta)
    ref = sched.step(o.cpu(), t, x.cpu(), eta=eta, variance_noise=nz.cpu()).prev_sample
    assert rel(out.cpu(), ref) < 2e-6, rel(out.cpu(), ref)


def _dpm_case(pt, n, k, seed):
    """drive the oracle scheduler (prediction_type pt) through steps 0..k with plausible outputs; the inputs and result of step k"""
    sched = DPMSolverMultistepScheduler(prediction_type=pt)
    sched.set_timesteps(n)
    ts, acp = sched.timesteps.tolist(), sched.alphas_cumprod
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(*SHAPE, generator=g) * 2 - 1
    for j in range(k + 1):
        a = acp[ts[j]]
        nz = torch.randn(*SHAPE, generator=g)
        x = a.sqrt() * x0 + (1 - a).sqrt() * nz
        eps = nz + 0.1 * torch.randn(*SHAPE, generator=g)
        x0_hat = (x - (1 - a).sqrt() * eps) / a.sqrt()
        o = {"sample": x0_hat, "v_prediction": a.sqrt() * eps - (1 - a).sqrt() * x0_hat}[pt]
        m_prev = sched.model_outputs[-1]
        out = sched.step(o, ts[j], x).prev_sample
    last = k == n - 1
    order = 1 if k == 0 or (last and n < 15) else 2
    acps = (float(acp[ts[k]]), float(acp[ts[k - 1]]) if order == 2 else 0.0, float(acp[0 if last else ts[k + 1]]))
    return x, o, m_prev, order, acps, out, sched.model_outputs[-1]


@pytest.mark.parametrize("pt", NON_EPS)
@pytest.mark.parametrize("n,k", [(20, 0), (20, 1), (20, 10), (20, 19), (5, 4)])
def test_dpmpp_step_pred_matches_scheduler(cuda, pt, n, k):
    x, o, m_prev, order, (a0, a1, at), ref, ref_m = _dpm_case(pt, n, k, 100 * n + k)
    x, o = x.to(cuda), o.to(cuda)
    hist = m_prev.to(cuda) if m_prev is not None else torch.full_like(x, float("nan"))
    out = torch.empty_like(x)
    _dpm_call(pt, o, x, hist, hist, None, None, out, 0, a0, a1, at, order)
    assert rel(out.cpu(), ref) < 2e-6, rel(out.cpu(), ref)
    assert rel(hist.cpu(), ref_m) < 2e-6, "the history buffer must hold this step's x0 prediction"


@pytest.mark.parametrize("pt", NON_EPS)
def test_step_pred_kernels_inpaint_prompt_frames(cuda, pt):
    """keep > 0: prompt frames are p_a prompt + p_b prompt_noise (DDPM: copied from `known`), every other frame is the step's own
    result bit for bit, and the DPM-Solver history keeps the model's prediction in the prompt frames too"""
    B, C, T = SHAPE
    keep = 7
    g = torch.Generator(device="cuda").manual_seed(3)
    prompt, pn = torch.rand(B, C, keep, device=cuda, generator=g) * 2 - 1, torch.randn(B, C, keep, device=cuda, generator=g)
    x, nz, m1 = (torch.randn(*SHAPE, device=cuda, generator=g) for _ in range(3))
    acp = DDIMScheduler().alphas_cumprod
    o = _output(pt, x, acp[500].to(cuda), g)
    pa, pb = 0.8, 0.6
    want = pa * prompt + pb * pn
    for kind in ("ddpm", "ddim", "dpmpp"):
        outs, hists = [], []
        for k, pp, pq in ((0, None, None), (keep, prompt, pn)):
            out, hist = torch.empty_like(x), m1.clone()
            if kind == "ddpm":
                known = torch.zeros_like(x)
                known[..., :keep] = want
                _ddpm_call(pt, o, x, nz, known if k else None, out, k, float(acp[500]), float(acp[490]))
            elif kind == "ddim":
                _ddim_call(pt, o, x, nz, pp, pq, out, k, float(acp[500]), float(acp[480]), 1.0, pa, pb)
            else:
                _dpm_call(pt, o, x, hist, hist, pp, pq, out, k, float(acp[500]), float(acp[550]), float(acp[450]), 2, pa, pb)
            outs.append(out)
            hists.append(hist)
        assert torch.equal(outs[1][..., keep:], outs[0][..., keep:]), kind
        assert rel(outs[1][..., :keep], want) < 1e-6, kind
        assert torch.equal(hists[1], hists[0]), kind


def test_epsilon_pred_entry_points_are_the_old_ones(cuda):
    """PT_PRED_EPSILON through the `_pred` entry points gives the same bits as the entry points without the suffix"""
    B, C, T = SHAPE
    keep = 5
    g = torch.Generator(device="cuda").manual_seed(4)
    x, e, nz, m1 = (torch.randn(*SHAPE, device=cuda, generator=g) for _ in range(4))
    prompt, pn = torch.rand(B, C, keep, device=cuda, generator=g), torch.randn(B, C, keep, device=cuda, generator=g)
    known = torch.randn(*SHAPE, device=cuda, generator=g)
    acp = DDIMScheduler().alphas_cumprod
    runs = []
    for name_pt in (None, "epsilon"):
        r = []
        for a, ap, noise, kn, k in ((float(acp[500]), float(acp[490]), nz, None, 0), (float(acp[10]), 1.0, None, known, keep)):
            out = torch.empty_like(x)
            _ddpm_call(name_pt, e, x, noise, kn, out, k, a, ap)
            r.append(out)
        for eta, k in ((0.0, 0), (1.0, keep)):
            out = torch.empty_like(x)
            _ddim_call(name_pt, e, x, nz, prompt if k else None, pn if k else None, out, k, float(acp[600]), float(acp[580]), eta, 0.7, 0.5)
            r.append(out)
        for order, k in ((1, 0), (2, keep)):
            out, hist = torch.empty_like(x), m1.clone()
            _dpm_call(name_pt, e, x, hist, hist, prompt if k else None, pn if k else None, out, k, float(acp[500]), float(acp[550]),
                      float(acp[450]), order, 0.7, 0.5)
            r += [out, hist]
        runs.append(r)
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- Gaussian target
@pytest.mark.parametrize("kind,eta,n", [("ddpm", None, 100), ("ddim", 0.0, 50), ("ddim", 1.0, 50), ("dpm", None, 20)])
def test_gaussian_target_kernel_loops_agree(cuda, kind, eta, n):
    """The samplers' own step code (`_step`, the fused kernels) driven by the exact predictor of x0 ~ N(0, 0.577^2), given as eps,
    x0 or v (computed in float64, rounded to fp32).  The three loops agree to 1e-5 (DESIGN section 5: an fp32 restatement of these
    steps keeps each parameterisation within 4e-7 of the float64 loop)."""
    _, model = so.load_model("tiny", cuda)
    B, C, T, s = 25, 8, 1000, 0.577
    g = torch.Generator(device="cuda").manual_seed(5)
    x_T = torch.randn(B, C, T, device=cuda, generator=g)
    noises = torch.randn(n, B, C, T, device=cuda, generator=g)
    res = {}
    for pt in PRED:
        smp = so.make_sampler(model, kind, eta, n, pt)
        x = x_T.clone()
        smp._T = T
        smp._static = {"eps": torch.empty_like(x)}
        smp._start(x, None, None, 0)
        acp = smp.acp.double().to(cuda)
        for i, t in enumerate(smp.timesteps):
            a, xd = acp[t], x.double()
            eps = (1 - a).sqrt() * xd / (a * s * s + 1 - a)
            x0 = (xd - (1 - a).sqrt() * eps) / a.sqrt()
            smp._static["eps"].copy_({"epsilon": eps, "sample": x0, "v_prediction": a.sqrt() * eps - (1 - a).sqrt() * x0}[pt])
            smp._step(i, t, x, noises, None)
        res[pt] = x
    e = {pt: rel(res[pt], res["epsilon"]) for pt in NON_EPS}
    print(f"\n[gaussian {kind} eta={eta} n={n}] vs epsilon loop: sample {e['sample']:.2e}, v {e['v_prediction']:.2e}; "
          f"std {res['epsilon'].std().item():.3f}")
    assert max(e.values()) < 1e-5, e
    assert 0.4 < res["epsilon"].std().item() < 0.8


# ---------------------------------------------------------------------------------------------------------------- training
def _oracle_train(cfg, model, inp, pt, gamma):
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point() and "inv_freq" not in k) for k, v in model.state_dict().items()}
    loss, _ = po.train_step_loss(sd, cfg, inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"], prediction_type=pt,
                                 snr_gamma=gamma)
    loss.backward()
    return loss.detach(), {k: v.grad for k, v in sd.items() if v.requires_grad and v.grad is not None and v.grad.abs().max() > 0}


# sizes: those of test_guidance_gpu.py's condition-dropout test (test_model_gpu.py gives the reason)
@pytest.mark.parametrize("gamma", [None, 5.0])
@pytest.mark.parametrize("pt", NON_EPS)
@pytest.mark.parametrize("cfg_name,B,T", [("tiny", 8, 64), ("mid", 2, 64)])
def test_train_step_prediction_type_matches_oracle(cuda, cfg_name, B, T, pt, gamma):
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model(cfg_name, cuda, train=True)
    inp = synth_inputs(cfg, B, T, seed=1, device=cuda)
    inp["t"][0] = 999
    ref_loss, ref_grads = _oracle_train(cfg, model, inp, pt, gamma)
    loss = DenoiserTrainStep(model, prediction_type=pt, snr_gamma=gamma)(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
    torch.cuda.synchronize()
    e_l, e_g = rel(loss, ref_loss), so.grad_err(model, ref_grads)
    print(f"\n[{cfg_name} {B}x{T} {pt} snr_gamma={gamma}] loss {e_l:.2e} global grad {e_g:.2e}")
    assert e_l < TOL and e_g < TOL, (e_l, e_g)


def test_train_step_graph_replays_fresh_timesteps(cuda):
    """the Min-SNR weight and the v target are formed on the device from t: replays of one captured step with two (t, noise) pairs
    equal eager steps with the same pairs"""
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 8, 64
    inp = synth_inputs(cfg, B, T, seed=4, device=cuda)
    stepper = DenoiserTrainStep(model, prediction_type="v_prediction", snr_gamma=5.0)
    t, noise = inp["t"].clone(), inp["noise"].clone()
    g = torch.Generator(device="cuda").manual_seed(8)
    pairs = [(inp["t"].clone(), inp["noise"].clone()),
             (torch.randint(0, 1000, (B,), device=cuda, generator=g), torch.randn(inp["noise"].shape, device=cuda, generator=g))]
    loss = torch.zeros((), device=cuda)
    named = list(model.named_parameters())

    def step():
        return stepper(inp["x0"], noise, t, inp["ids"], loss_out=loss)

    eager = []
    for tt, nn in pairs:
        t.copy_(tt)
        noise.copy_(nn)
        step()
        torch.cuda.synchronize()
        eager.append((float(loss), torch.cat([p.grad.flatten() for _, p in named if p.grad is not None]).clone()))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for (tt, nn), (l_e, g_e) in zip(pairs, eager):
        t.copy_(tt)
        noise.copy_(nn)
        graph.replay()
        torch.cuda.synchronize()
        gr = torch.cat([p.grad.flatten() for _, p in named if p.grad is not None])
        assert abs(float(loss) - l_e) <= 1e-3 * abs(l_e) and rel(gr, g_e) < 1e-3
    assert abs(eager[0][0] - eager[1][0]) > 1e-3 * abs(eager[0][0]), "the two pairs must give different losses"


# ---------------------------------------------------------------------------------------------------------------- sampling loops
@pytest.fixture(scope="module")
def tiny(cuda):
    return so.load_model("tiny", cuda)


def _bound(model, cfg, kind, eta, n_infer, pt, w, inp, x_T, noises, want, prompt=None, pn=None):
    """what the fp32 oracle loop makes of the 2e-2 per-call bar (DESIGN section 5), and at least that bar doubled (the bound of the
    stochastic loops in test_fast_sampler_gpu.py)"""
    e = rel(so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, pt=pt, w=w, prompt=prompt, prompt_noise=pn,
                           eps_err=TOL, err_seed=29), want)
    return max(e, 2 * TOL)


KINDS = [("ddpm", None), ("ddim", 0.0), ("ddim", 1.0), ("dpm", None)]


@pytest.mark.parametrize("pt", NON_EPS)
@pytest.mark.parametrize("kind,eta", KINDS)
def test_sampler_loop_matches_oracle(cuda, tiny, kind, eta, pt):
    cfg, model = tiny
    B, T, n_infer = 2, 16, 5
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 5, cuda)
    outs = {gr: so.make_sampler(model, kind, eta, n_infer, pt, gr).sample(inp["ids"], T, x_T=x_T, noises=noises)
            for gr in (False, True)}
    # GroupNorm statistics are accumulated with fp32 atomics (order not fixed), so two runs agree to rounding, not bit for bit
    assert rel(outs[False], outs[True]) < 1e-3, "graph replay must reproduce the eager loop"
    want = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, pt=pt)
    eps_loop = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises)
    bound = _bound(model, cfg, kind, eta, n_infer, pt, None, inp, x_T, noises, want)
    e = {gr: rel(outs[gr], want) for gr in (False, True)}
    print(f"\n[{kind} eta={eta} {pt} tiny, {n_infer} steps] rel err vs fp32 oracle loop: graph {e[True]:.2e}, eager {e[False]:.2e} "
          f"(bound {bound:.2e}; vs the epsilon reading of the same model {rel(want, eps_loop):.2e})")
    assert e[True] < bound and e[False] < bound, (e, bound)


@pytest.mark.parametrize("pt", NON_EPS)
def test_guided_sampler_loop_matches_oracle(cuda, tiny, pt):
    cfg, model = tiny
    B, T, n_infer, w = 2, 16, 5, 3.0
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 6, cuda)
    got = so.make_sampler(model, "ddim", 0.0, n_infer, pt).sample(inp["ids"], T, x_T=x_T, noises=noises, guidance_scale=w)
    want = so.oracle_loop(model, cfg, "ddim", 0.0, n_infer, inp["ids"], x_T, noises, pt=pt, w=w)
    bound = _bound(model, cfg, "ddim", 0.0, n_infer, pt, w, inp, x_T, noises, want)
    print(f"\n[guided ddim {pt} w={w}] rel err {rel(got, want):.2e} (bound {bound:.2e})")
    assert rel(got, want) < bound


@pytest.mark.parametrize("pt", NON_EPS)
@pytest.mark.parametrize("kind,eta", [("ddpm", None), ("dpm", None)])
def test_sampler_prompt_inpainting_matches_oracle(cuda, tiny, kind, eta, pt):
    cfg, model = tiny
    B, T, P, n_infer = 2, 16, 6, 4
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 7, cuda)
    prompt = inp["x0"][..., :P].contiguous()
    g = torch.Generator(device="cuda").manual_seed(13)
    pn = torch.randn(n_infer, B, cfg["in_channels"], P, device=cuda, generator=g)
    got = so.make_sampler(model, kind, eta, n_infer, pt).sample(inp["ids"], T, x_T=x_T, noises=noises, prompt=prompt, prompt_noise=pn)
    want = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, pt=pt, prompt=prompt, prompt_noise=pn)
    bound = _bound(model, cfg, kind, eta, n_infer, pt, None, inp, x_T, noises, want, prompt, pn)
    print(f"\n[{kind} {pt} + prompt] rel err {rel(got, want):.2e} (bound {bound:.2e})")
    assert torch.equal(got[..., :P], prompt), "the prompt frames must come out clean"
    assert rel(got, want) < bound


# ---------------------------------------------------------------------------------------------------------------- launches
def _count(fn, monkeypatch):
    """kernel launches of fn() and the entry points it called"""
    from prompt_tts_b200 import _lib, ops
    names = []
    real = ops.call

    def rec(name, *args):
        names.append(name)
        return real(name, *args)

    monkeypatch.setattr(ops, "call", rec)
    torch.cuda.synchronize()
    l0 = _lib.lib().pt_launch_count()
    fn()
    torch.cuda.synchronize()
    n = _lib.lib().pt_launch_count() - l0
    monkeypatch.setattr(ops, "call", real)
    return n, names


def test_launch_counts(cuda, monkeypatch):
    """The default train step still launches add_noise + mse_fwd_bwd, a non-default one add_noise + diffusion_loss: the same count.
    Every sampler calls its `_pred` step entry point once per step whatever the type, and launches as many kernels for each type."""
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 8, 64
    inp = synth_inputs(cfg, B, T, seed=9, device=cuda)
    counts = {}
    for pt, gamma in (("epsilon", None), ("v_prediction", None), ("sample", 5.0), ("epsilon", 5.0)):
        stepper = DenoiserTrainStep(model, prediction_type=pt, snr_gamma=gamma)
        stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"])            # first-use work outside the counted call
        n, names = _count(lambda: stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"]), monkeypatch)
        default = pt == "epsilon" and gamma is None
        assert ("mse_fwd_bwd" in names) == default and ("diffusion_loss" in names) != default, (pt, gamma, names)
        counts[(pt, gamma)] = n
    assert len(set(counts.values())) == 1, counts
    model.eval()
    T, n_infer = 16, 3
    inp = synth_inputs(cfg, 2, T, seed=10, device=cuda)
    for kind, eta, step in (("ddpm", None, "ddpm_step"), ("ddim", 1.0, "ddim_step"), ("dpm", None, "dpmpp_step")):
        c = {}
        for pt in PRED:
            smp = so.make_sampler(model, kind, eta, n_infer, pt)
            smp.sample(inp["ids"], T, seed=1)
            n, names = _count(lambda: smp.sample(inp["ids"], T, seed=1), monkeypatch)
            want = step + "_pred"
            assert names.count(want) == n_infer and not any(s.startswith(step) and s != want for s in names), (kind, pt, names)
            c[pt] = n
        assert len(set(c.values())) == 1, (kind, c)
