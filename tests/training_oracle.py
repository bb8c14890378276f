"""The train-step tests' shared oracle and harness: one fp32 autograd step of tests/prediction_oracle.py's train_step_loss on the
model's weights, the flat gradient vector, CUDA-graph capture, the model / stepper / optimiser set-up and the two-rank launcher of
tests/dp_worker.py."""
import json
import os
import subprocess
import sys

import pytest
import torch

import prediction_oracle as po
import ref_model
from util import ROOT, load_model, rel, synth_inputs

# lr large enough that a few steps move the weights measurably; the clip threshold below the gradient norm, so clipping is active
OPT_KW = dict(lr=1e-3, betas=(0.95, 0.999), weight_decay=1e-2, eps=1e-8, max_norm=0.05)


def oracle_params(model):
    """a leaf copy of the model's state_dict: every floating-point tensor but the rotary inv_freq buffers requires grad"""
    return {k: v.detach().clone().requires_grad_(v.is_floating_point() and "inv_freq" not in k) for k, v in model.state_dict().items()}


def oracle_train(cfg, model, inp, *, prediction_type="epsilon", snr_gamma=None, cond_keep=None, autocast=False):
    """fp32 autograd of prediction_oracle.train_step_loss on the model's weights and a synth_inputs batch: x_t, the prediction, the
    loss and the gradient of every parameter that requires grad (None where autograd did not reach it).  autocast: the forward
    under torch.autocast(bf16) and the loss in fp32, the reference's own bf16 path."""
    sd = oracle_params(model)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        loss, pred = po.train_step_loss(sd, cfg, inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"],
                                        prediction_type=prediction_type, snr_gamma=snr_gamma, cond_keep=cond_keep)
    loss.backward()
    xt = ref_model.add_noise(inp["x0"], inp["noise"], inp["t"])
    return xt, pred.detach(), loss.detach(), {k: v.grad for k, v in sd.items() if v.requires_grad}


def flat_grads(model):
    """the model's gradients, concatenated in parameter order"""
    return torch.cat([p.grad.flatten() for p in model.parameters() if p.grad is not None])


def capture(fn):
    """fn() once on a side stream, as torch asks before capture, then a CUDA graph of fn()"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def check_replays_fresh_inputs(model, step, static, inputs):
    """step(loss) reads its inputs from the buffers of `static` and writes its loss into `loss`.  With each entry of `inputs`
    copied into those buffers: one eager step, then one replay of a captured step, which must give the same loss and flat gradient
    (to 1e-3: GroupNorm statistics are accumulated with fp32 atomics).  Returns the eager (loss, flat gradient) of each entry."""
    loss = torch.zeros((), device=static[0].device)

    def load(x):
        for buf, v in zip(static, x):
            buf.copy_(v)

    eager = []
    for x in inputs:
        load(x)
        step(loss)
        torch.cuda.synchronize()
        eager.append((float(loss), flat_grads(model)))
    graph = capture(lambda: step(loss))
    for x, (l_e, g_e) in zip(inputs, eager):
        load(x)
        graph.replay()
        torch.cuda.synchronize()
        assert abs(float(loss) - l_e) <= 1e-3 * abs(l_e) and rel(flat_grads(model), g_e) < 1e-3
    return eager


def setup(cuda, cfg_name="tiny", B=2, T=16, accumulation_steps=1, ema_kw=None):
    """load_model's weights, a seeded batch, a DenoiserTrainStep, a FusedClipAdamW with OPT_KW and, for ema_kw not None, a
    FusedEMA with ema_kw"""
    from prompt_tts_b200.optim import FusedClipAdamW, FusedEMA
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = load_model(cfg_name, cuda, train=True)
    inp = synth_inputs(cfg, B, T, seed=2, device=cuda)
    stepper = DenoiserTrainStep(model, accumulation_steps=accumulation_steps)
    opt = FusedClipAdamW(stepper, **OPT_KW)
    ema = FusedEMA(opt, **ema_kw) if ema_kw is not None else None
    return cfg, model, inp, stepper, opt, ema


def run_two_ranks(mode, cfg, B, T, port):
    """tests/dp_worker.py in `mode` on two GPUs, one process per GPU over NCCL, launched the way the bench is launched; rank 0's
    result"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "dp_worker.py"), mode, cfg, str(B), str(T)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1][len("RESULT "):])
    print(res)
    return res
