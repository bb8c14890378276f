"""GPU: the EMA of the weights (`optim.FusedEMA`) against the diffusers 0.15 `EMAModel` restatement (oracle/diffusers_shim) stepped on
the same parameters -- the fused kernel, the device-side decay schedule, eager and captured training, `swapped()`, checkpoints,
the launch count and two data-parallel ranks.

Two forward/backward passes of the train step are not bit-identical (GroupNorm statistics and weight gradients are accumulated with
fp32 atomics), so where two runs are compared bit for bit the second one is fed the gradients the first one computed: what is
compared is the optimiser and the EMA, which are deterministic."""
import math
import os
import sys

import pytest
import torch

import training_oracle as to
from util import ROOT, load_model, rel

sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))
from diffusers.training_utils import EMAModel  # noqa: E402

pytestmark = pytest.mark.gpu
# warmup: the device's double pow() and the host's may differ in the last bits of 1 - (1 + step / inv_gamma) ** -power (CUDA
# documents pow to 2 ulp, glibc to 1).  Near decay ~ 1 that is a few ulp of 1.0 in the decay, and at most one fp32 ulp in the
# coefficient 1 - decay when it falls on a rounding boundary; over a few steps the average then differs by far less than this.
WARMUP_DECAY_ATOL = 2.0 ** -50
WARMUP_EMA_REL = 1e-6
VARIANTS = {"default": {}, "update_after_step=2": dict(update_after_step=2), "min_decay=0.5": dict(decay=0.9, min_decay=0.5),
            "warmup": dict(use_ema_warmup=True, inv_gamma=1.0, power=2 / 3)}


def _run(stepper, inp, sl=slice(None)):
    stepper(inp["x0"][sl], inp["noise"][sl], inp["t"][sl], inp["ids"][sl], inp["mask"][sl])


def _check_against_shim(model, ema, shim, exact=True):
    sd = ema.model_state_dict()
    msd = model.state_dict()
    assert list(sd) == list(msd) and all(sd[k].shape == msd[k].shape for k in msd)
    params = dict(model.named_parameters())
    for (k, _), s in zip(model.named_parameters(), shim.shadow_params):
        if exact:
            assert torch.equal(sd[k], s), (k, int((sd[k] != s).sum()))
        else:
            assert rel(sd[k], s) <= WARMUP_EMA_REL, (k, rel(sd[k], s))
    for k in msd:
        if k not in params:
            assert torch.equal(sd[k], msd[k]), k          # buffers come from the model
    assert ema.optimization_step == shim.optimization_step
    d = float(ema.cur_decay)
    assert d == shim.cur_decay_value if exact else abs(d - shim.cur_decay_value) <= WARMUP_DECAY_ATOL


# ------------------------------------------------------------------------------------------------ 1. the fused kernel
@pytest.mark.parametrize("g_bf16", [False, True])
def test_fused_kernel_equals_plain_step_and_torch_update(cuda, g_bf16):
    from prompt_tts_b200 import ops, optim as O
    n = 4 * 250_007
    gen = torch.Generator(device=cuda).manual_seed(11)
    p = torch.randn(n, device=cuda, generator=gen)
    g = torch.randn(n, device=cuda, generator=gen) * 1e-2
    g = g.to(torch.bfloat16) if g_bf16 else g
    m = torch.randn(n, device=cuda, generator=gen) * 1e-3
    v = torch.rand(n, device=cuda, generator=gen) * 1e-4
    e = p + torch.randn(n, device=cuda, generator=gen) * 1e-2
    host = [0.0] * O.NSTATE
    host[O.LR], host[O.BETA1], host[O.BETA2], host[O.EPS], host[O.WD], host[O.MAX_NORM], host[O.GSCALE] = 1e-3, 0.95, 0.999, 1e-8, 1e-2, 1.0, 1.0
    st = torch.tensor(host, device=cuda)
    gsq = (g.float() ** 2).sum().reshape(1)
    ops.call("adamw_prepare", ops._p(st), ops._p(gsq), ops._stream())
    est = torch.zeros(O.EMA_NSTATE, dtype=torch.float64, device=cuda)
    est[O.EMA_DECAY], est[O.EMA_INV_GAMMA], est[O.EMA_POWER], est[O.EMA_STEP] = 0.9999, 1.0, 2 / 3, 999.0
    ops.call("ema_prepare", ops._p(est), ops._stream())
    c = float(est[O.EMA_COEF])
    assert float(est[O.EMA_CUR_DECAY]) == 1000 / 1009 and c == float(torch.tensor(1 - 1000 / 1009, dtype=torch.float32))
    p1, m1, v1, w1 = p.clone(), m.clone(), v.clone(), torch.zeros(n, dtype=torch.bfloat16, device=cuda)
    ops.call("adamw_step_dev", ops._p(p1), ops._p(g), int(g_bf16), ops._p(m1), ops._p(v1), ops._p(w1), n, ops._p(st), ops._stream())
    p2, m2, v2, w2, e2 = p.clone(), m.clone(), v.clone(), torch.zeros(n, dtype=torch.bfloat16, device=cuda), e.clone()
    ops.call("adamw_ema_step_dev", ops._p(p2), ops._p(g), int(g_bf16), ops._p(m2), ops._p(v2), ops._p(w2), ops._p(e2), n, ops._p(st),
             ops._p(est), ops._stream())
    assert not torch.equal(p1, p) and torch.equal(p1, p2) and torch.equal(m1, m2) and torch.equal(v1, v2) and torch.equal(w1, w2)
    want = e.clone()
    want.sub_(c * (want - p1))
    assert torch.equal(e2, want), int((e2 != want).sum())
    # the swap: one pass, bf16 shadow of the new masters
    ops.call("ema_swap", ops._p(p2), ops._p(e2), ops._p(w2), n, ops._stream())
    assert torch.equal(p2, want) and torch.equal(e2, p1) and torch.equal(w2, want.to(torch.bfloat16))


# ------------------------------------------------------------------------------------------------ 2. the decay schedule
@pytest.mark.parametrize("kw", [dict(), dict(decay=0.9, update_after_step=3), dict(decay=0.95, min_decay=0.5), dict(decay=1.0),
                                dict(use_ema_warmup=True), dict(use_ema_warmup=True, inv_gamma=3.0, power=0.75, decay=0.95)],
                         ids=["default", "update_after", "min_decay", "decay1", "warmup", "warmup_cap"])
def test_device_decay_schedule_matches_shim(cuda, kw):
    from prompt_tts_b200 import ops, optim as O
    shim = EMAModel([], **kw)
    full = {**dict(decay=0.9999, min_decay=0.0, update_after_step=0, use_ema_warmup=False, inv_gamma=1.0, power=2 / 3), **kw}
    est = torch.zeros(O.EMA_NSTATE, dtype=torch.float64, device=cuda)
    est[O.EMA_DECAY], est[O.EMA_MIN_DECAY], est[O.EMA_UPDATE_AFTER] = full["decay"], full["min_decay"], full["update_after_step"]
    est[O.EMA_USE_WARMUP], est[O.EMA_INV_GAMMA], est[O.EMA_POWER] = float(full["use_ema_warmup"]), full["inv_gamma"], full["power"]
    worst = 0.0
    for k in range(1, 201):
        ops.call("ema_prepare", ops._p(est), ops._stream())
        got = est.tolist()
        want = shim.get_decay(k)
        assert got[O.EMA_STEP] == k
        c_want = float(torch.tensor(1 - want, dtype=torch.float32))
        if full["use_ema_warmup"]:
            worst = max(worst, abs(got[O.EMA_CUR_DECAY] - want))
            assert abs(got[O.EMA_CUR_DECAY] - want) <= WARMUP_DECAY_ATOL, (k, got[O.EMA_CUR_DECAY], want)
            assert abs(got[O.EMA_COEF] - c_want) <= math.ulp(c_want) * 2 ** 29, (k, got[O.EMA_COEF], c_want)      # one fp32 ulp
        else:
            assert got[O.EMA_CUR_DECAY] == want and got[O.EMA_COEF] == c_want, (k, got[O.EMA_CUR_DECAY], want)
    print(f"{kw}: worst |device decay - host decay| = {worst:.3g}")


# ------------------------------------------------------------------------------------------------ 3. eager training, end to end
@pytest.mark.parametrize("cfg_name", ["tiny", "mid"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_ema_matches_shim_end_to_end(cuda, cfg_name, variant):
    from prompt_tts_b200.models import TTSSingleSpeaker
    kw = VARIANTS[variant]
    cfg, model, inp, stepper, opt, ema = to.setup(cuda, cfg_name, ema_kw=kw)
    shim = EMAModel(model.parameters(), **kw)
    for _ in range(5):
        _run(stepper, inp)
        opt.step()
        shim.step(model.parameters())
        _check_against_shim(model, ema, shim, exact=variant != "warmup")
    assert ema.optimization_step == 5 and opt.step_count == 5
    fresh = TTSSingleSpeaker(cfg).to(cuda)
    fresh.load_state_dict(ema.model_state_dict(), strict=True)
    # the EMA moved away from both the initial and the trained weights, and proj_out (never trained) kept its value
    sd = ema.model_state_dict()
    k = next(k for k, p in model.named_parameters() if p.dim() >= 2 and "proj_out" not in k)
    assert not torch.equal(sd[k], model.state_dict()[k])
    for k in ema.frozen:
        assert torch.equal(sd[k], model.state_dict()[k])


def test_ema_constructed_after_attach_starts_from_current_weights(cuda):
    from prompt_tts_b200.optim import FusedEMA
    cfg, model, inp, stepper, opt, _ = to.setup(cuda)
    for _ in range(2):
        _run(stepper, inp)
        opt.step()
    ema = FusedEMA(opt)
    assert torch.equal(ema.eflat, opt.pflat) and ema.optimization_step == 0
    shim = EMAModel(model.parameters())
    _run(stepper, inp)
    opt.step()
    shim.step(model.parameters())
    _check_against_shim(model, ema, shim)


# ------------------------------------------------------------------------------------------------ 4. graph capture
def test_ema_graph_replays(cuda):
    """One captured `step(); opt.step()` replayed: the EMA's step counter and decay live in device memory, so every replay is the
    next EMA step."""
    cfg, model, inp, stepper, opt, ema = to.setup(cuda, ema_kw={})
    shim = EMAModel(model.parameters())

    def full():
        _run(stepper, inp)
        opt.step()

    full()                                  # eager step 1 (defines the flat layout, starts the average)
    shim.step(model.parameters())
    g = to.capture(full)                    # eager step 2 on the side stream, then the capture (which runs nothing)
    shim.step(model.parameters())
    _check_against_shim(model, ema, shim)
    for _ in range(5):
        g.replay()
        torch.cuda.synchronize()
        shim.step(model.parameters())
        _check_against_shim(model, ema, shim)
    assert ema.optimization_step == 7 and opt.step_count == 7


def test_ema_steps_once_per_accumulation_window_in_a_graph(cuda):
    cfg, model, inp, stepper, opt, ema = to.setup(cuda, B=4, accumulation_steps=2, ema_kw=dict(decay=0.9))
    shim = EMAModel(model.parameters(), decay=0.9)

    def window():
        for half in (slice(0, 2), slice(2, 4)):
            _run(stepper, inp, half)
            opt.step()

    window()
    shim.step(model.parameters())
    g = to.capture(window)
    shim.step(model.parameters())           # the warm-up window
    _check_against_shim(model, ema, shim)
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        shim.step(model.parameters())
        _check_against_shim(model, ema, shim)
    assert ema.optimization_step == 5 and opt.step_count == 5


# ------------------------------------------------------------------------------------------------ 5. swapped()
def test_swapped_samples_the_ema_and_restores_everything(cuda):
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.sample import DDIMSampler
    cfg, model, inp, stepper, opt, ema = to.setup(cuda, ema_kw=dict(decay=0.9))
    for _ in range(3):
        _run(stepper, inp)
        opt.step()
    gfix = stepper.grad_sync.flat.clone()           # the last step's gradients, fed to every replay below (module docstring)

    def train():
        _run(stepper, inp)
        stepper.grad_sync.flat.copy_(gfix)
        opt.step()

    g = to.capture(train)                           # a training graph captured before the swap
    torch.cuda.synchronize()
    bufs = lambda: [opt.pflat, opt.wflat, opt.m, opt.v, ema.eflat, opt.state, ema.state]     # noqa: E731
    before = [b.clone() for b in bufs()]
    assert not torch.equal(opt.pflat, ema.eflat)
    x_T = torch.randn(2, cfg["in_channels"], 16, device=cuda, generator=torch.Generator(device=cuda).manual_seed(5))
    ema_sd = ema.model_state_dict()
    with ema.swapped():
        assert torch.equal(opt.pflat, before[4]) and torch.equal(ema.eflat, before[0])
        assert torch.equal(opt.wflat, opt.pflat.to(torch.bfloat16))
        assert all(torch.equal(model.state_dict()[k], v) for k, v in ema_sd.items())
        with pytest.raises(_lib.PtError, match="swapped"):
            opt.step()
        with pytest.raises(_lib.PtError, match="swapped"):
            ema.model_state_dict()
        got = DDIMSampler(model, n_infer=3).sample(inp["ids"], 16, x_T=x_T)
    for b, w in zip(bufs(), before):
        assert torch.equal(b, w)
    _, fresh = load_model("tiny", cuda, train=True, seed=9)
    fresh.load_state_dict(ema_sd, strict=True)
    want = DDIMSampler(fresh, n_infer=3).sample(inp["ids"], 16, x_T=x_T)
    assert torch.equal(got, want), rel(got, want)
    # the graph captured before the swap still trains the right buffers: equal to a twin run from the same state without a swap
    for _ in range(2):
        g.replay()
    after_swap = [b.clone() for b in bufs()]
    for b, w in zip(bufs(), before):
        b.copy_(w)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    for b, w in zip(bufs(), after_swap):
        assert torch.equal(b, w)
    assert ema.optimization_step == 6 and not torch.equal(ema.eflat, before[4])


def test_swapped_refuses_capture_and_copy_to_is_permanent(cuda):
    from prompt_tts_b200 import _lib
    cfg, model, inp, stepper, opt, ema = to.setup(cuda, ema_kw=dict(decay=0.9))
    for _ in range(2):
        _run(stepper, inp)
        opt.step()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with pytest.raises(_lib.PtError, match="captured"):
        with torch.cuda.graph(g):
            with ema.swapped():
                pass
    assert not ema.is_swapped
    sd = ema.model_state_dict()
    ema.copy_to()
    assert torch.equal(opt.pflat, ema.eflat) and torch.equal(opt.wflat, opt.pflat.to(torch.bfloat16))
    assert all(torch.equal(model.state_dict()[k], v) for k, v in sd.items())


# ------------------------------------------------------------------------------------------------ 6. resume
def test_resume_is_bit_identical(cuda):
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.optim import FusedClipAdamW, FusedEMA
    from prompt_tts_b200.train import DenoiserTrainStep
    ema_kw = dict(decay=0.95, update_after_step=1, min_decay=0.1)
    cfg, model, inp, stepper, opt, ema = to.setup(cuda, ema_kw=ema_kw)
    for _ in range(3):
        _run(stepper, inp)
        opt.step()
    ck = ({k: v.clone() for k, v in model.state_dict().items()}, opt.state_dict(), ema.state_dict())
    grads = []
    for _ in range(2):
        _run(stepper, inp)
        grads.append(stepper.grad_sync.flat.clone())
        opt.step()
    torch.cuda.synchronize()
    # resume into fresh objects (other initial weights, default EMA hyper-parameters: the checkpoint's are restored)
    _, model2 = load_model("tiny", cuda, train=True, seed=5)
    model2.load_state_dict(ck[0], strict=True)
    stepper2 = DenoiserTrainStep(model2)
    opt2 = FusedClipAdamW(stepper2, **to.OPT_KW)
    ema2 = FusedEMA(opt2)
    for k in range(2):
        _run(stepper2, inp)
        if k == 0:
            opt2.load_state_dict(ck[1])
            ema2.load_state_dict(ck[2])
            assert ema2.optimization_step == 3 and (ema2.decay, ema2.update_after_step, ema2.min_decay) == (0.95, 1, 0.1)
        stepper2.grad_sync.flat.copy_(grads[k])         # the gradients of the uninterrupted run (module docstring)
        opt2.step()
    for a, b in ((opt.pflat, opt2.pflat), (opt.wflat, opt2.wflat), (opt.m, opt2.m), (opt.v, opt2.v), (opt.state, opt2.state),
                 (ema.eflat, ema2.eflat), (ema.state, ema2.state)):
        assert torch.equal(a, b)
    s1, s2 = ema.model_state_dict(), ema2.model_state_dict()
    assert all(torch.equal(s1[k], s2[k]) for k in s1)
    bad = dict(ck[2], layout=ck[2]["layout"][1:])
    with pytest.raises(_lib.PtError, match="layout"):
        ema2.load_state_dict(bad)


# ------------------------------------------------------------------------------------------------ 7. launches
def test_opt_step_launch_count(cuda):
    from prompt_tts_b200 import _lib
    lib = _lib.lib()
    counts = {}
    for with_ema in (False, True):
        cfg, model, inp, stepper, opt, ema = to.setup(cuda, ema_kw={} if with_ema else None)
        _run(stepper, inp)
        opt.step()                              # attach (one cast of the shadow) happens here
        _run(stepper, inp)
        l0 = lib.pt_launch_count()
        opt.step()
        counts[with_ema] = lib.pt_launch_count() - l0
    assert counts == {False: 3, True: 4}, counts


# ------------------------------------------------------------------------------------------------ 8. two ranks
def test_two_rank_ema_identical(cuda):
    res = to.run_two_ranks("ema", "tiny3", 2, 64, 29543)
    for mode in ("fp32", "bf16"):
        assert res[mode]["optimization_step"] == 3
        assert res[mode]["ema_identical_on_all_ranks"] and res[mode]["weights_identical_on_all_ranks"], res
        assert res[mode]["ema_moved"], res
