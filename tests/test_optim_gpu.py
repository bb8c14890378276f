"""GPU: the fused clip + AdamW step (SURVEY 8f rank 1) against torch's clip_grad_norm_ + AdamW -- the reference's optimiser
lines train.py:41-47,116-120 -- applied to the same gradients, eagerly and replayed from a CUDA graph; gradient accumulation
(train.py:27,80); the bf16 shadow weights follow load_state_dict; input dtypes are converted, not misread."""
import pytest
import torch

import training_oracle as to
from util import load_model, rel

pytestmark = pytest.mark.gpu
KW = {k: v for k, v in to.OPT_KW.items() if k != "max_norm"}           # torch's AdamW takes no clip threshold


class TorchRef:
    """torch.optim.AdamW + clip_grad_norm_ on CPU copies, fed with the gradients the B200 step produced."""

    def __init__(self, model, max_norm):
        self.p = {k: p.detach().clone().cpu().contiguous().requires_grad_(True) for k, p in model.named_parameters()}
        self.opt = torch.optim.AdamW(list(self.p.values()), **KW)
        self.max_norm = max_norm

    def step(self, model):
        for k, p in model.named_parameters():
            self.p[k].grad = p.grad.detach().cpu().contiguous().clone() if p.grad is not None else None
        live = [q for q in self.p.values() if q.grad is not None]
        tn = torch.nn.utils.clip_grad_norm_(live, self.max_norm)
        self.opt.step()
        return float(tn)

    def worst(self, model):
        return max(rel(p.detach().cpu(), self.p[k]) for k, p in model.named_parameters())


def test_fused_clip_adamw_matches_torch(cuda):
    cfg, model, inp, stepper, opt, _ = to.setup(cuda)
    ref = TorchRef(model, 0.05)
    for it in range(3):
        stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
        tn = ref.step(model)
        gsq = opt.step()
        assert abs(float(gsq) ** 0.5 - tn) / tn < 1e-4
        assert tn > 0.05, "the test must exercise the clipping branch"
    assert opt.step_count == 3
    assert ref.worst(model) < 1e-5, ref.worst(model)
    # state_dict still has the reference layout (k=3 conv weights are permuted views of tap-major storage) and reads the master buffer
    sd = model.state_dict()
    named = dict(model.named_parameters())
    assert all(sd[k].shape == named[k].shape and torch.equal(sd[k].cpu(), named[k].detach().cpu()) for k in named)
    w = named["unet.mid_block.resnets.0.conv1.weight"]
    assert w.shape[2] == 3 and not w.is_contiguous() and w.permute(0, 2, 1).is_contiguous()
    # the GEMM operands are the optimiser's bf16 shadow: equal to bf16(master) in the GEMM layout, written by the AdamW kernel
    assert torch.equal(opt.wflat, opt.pflat.to(torch.bfloat16))
    # and the next forward uses the updated weights: loss changes
    l0 = float(stepper.loss)
    l1 = float(stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"]))
    assert l1 != l0 and abs(l1 - l0) / l0 < 0.5


def test_fused_adamw_graph_replays(cuda):
    """One captured `step(); opt.step()` replayed: the step counter / bias corrections / clip factor / learning rate live in device
    memory, so every replay is the next optimiser step (round 1 baked step = 2 into the graph: updates ~0.46x the correct size)."""
    cfg, model, inp, stepper, opt, _ = to.setup(cuda)
    ref = TorchRef(model, 0.05)

    def full():
        stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
        opt.step()

    stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])      # eager step 1 (defines the flat layout)
    ref.step(model)
    opt.step()
    g = to.capture(full)
    ref.step(model)                       # the warm-up step's gradients: opt.step() leaves param.grad as it is
    for it in range(5):
        if it == 3:                       # an LR scheduler writes the device-side learning rate between replays
            opt.set_lr(5e-4)
            for grp in ref.opt.param_groups:
                grp["lr"] = 5e-4
        g.replay()
        torch.cuda.synchronize()
        ref.step(model)                   # param.grad holds the gradients this replay computed (before its update)
        assert ref.worst(model) < 1e-5, (it, ref.worst(model))
    assert opt.step_count == 7
    assert torch.equal(opt.wflat, opt.pflat.to(torch.bfloat16))


def test_gradient_accumulation_matches_one_big_batch(cuda):
    """Two micro-batches under accumulation_steps = 2 (`accelerator.accumulate`, train.py:27,80) == one step on the concatenated batch."""
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model, inp, stepper, opt, _ = to.setup(cuda, B=4, T=32)
    big = DenoiserTrainStep(model)
    big(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
    g_big = big.grad_sync.flat.clone()
    acc = DenoiserTrainStep(model, accumulation_steps=2)
    flags = []
    for half in (slice(0, 2), slice(2, 4)):
        acc(inp["x0"][half], inp["noise"][half], inp["t"][half], inp["ids"][half], inp["mask"][half])
        flags.append(acc.sync_gradients)
    assert flags == [False, True]
    assert acc.grad_sync.groups == big.grad_sync.groups or [g[1:] for g in acc.grad_sync.groups] == [g[1:] for g in big.grad_sync.groups]
    assert rel(acc.grad_sync.flat, g_big) < 2e-3      # same per-sample bf16 arithmetic; GroupNorm / batch-shaped tiles differ in fp32 summation order only
    # the window starts from zero: a third micro-step does not see the previous window's sum
    acc(inp["x0"][:2], inp["noise"][:2], inp["t"][:2], inp["ids"][:2], inp["mask"][:2])
    assert not acc.sync_gradients and acc.grad_sync.flat.norm() < 0.9 * g_big.norm() * 2


def test_shadow_follows_load_state_dict_and_dtypes_are_converted(cuda):
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model, inp, stepper, opt, _ = to.setup(cuda)
    stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
    opt.step()
    _, other = load_model("tiny", cuda, train=True, seed=7)
    want = float(DenoiserTrainStep(other)(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"]))
    model.load_state_dict(other.state_dict())            # in-place writes into the flat master buffer, from outside the optimiser
    got = float(stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"]))
    assert abs(got - want) / want < 1e-5, (got, want)
    # int64 token ids / int32 timesteps / fp64 latents are converted at entry (the kernels read raw int32 / int64 / fp32 pointers)
    got2 = float(stepper(inp["x0"].double(), inp["noise"], inp["t"].to(torch.int32), inp["ids"].long(), inp["mask"]))
    assert got2 == got
    # optimiser checkpoints round-trip
    sd = opt.state_dict()
    opt.load_state_dict(sd)
    assert opt.step_count == 1
