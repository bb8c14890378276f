"""Parity of the B200 path against the CPU/GPU-fp32 oracle restatement (oracle/ref_model.py) on identical seeded
inputs and an identical state_dict.  Tolerance: north-star 2e-2 relative (bf16 compute) on outputs and gradients."""
import pytest
import torch

import training_oracle as to
from util import load_model, rel, synth_inputs

pytestmark = pytest.mark.gpu
TOL = 2e-2


# Sizes: the two toy configs at >= 272 (batch x frame) positions, `mid` = the real level-0/1 widths (320 / 640 channels, head dims
# 40 / 80, GroupNorm groups of 10 / 20 channels, 768-d text context) and `1d_config` = BASELINE.json's model at B = 2, T = 752
# (4 levels, head dims 40 / 80 / 160, Lk = 550, stream-K weight gradients).  Measured on B200 (gpurun_out/r2a, r2b; out / global
# gradient): tiny 8x64 1.2e-2 / 1.0e-2, tiny3 2x136 1.2e-2 / 1.4e-2, tiny3 8x128 1.3e-2 / 0.9e-2, mid 2x64 1.1e-2 / 1.1e-2,
# 1d_config 2x752 1.1e-2 / 0.8e-2.  With fewer than ~100 positions per weight-gradient sum (tiny3 3x32: 2.07e-2, tiny 2x16: 1.95e-2;
# the reference's own torch.autocast(bf16) run: 2.30e-2 / 2.45e-2) bf16 rounding noise does not average out and NO bf16 path meets
# 2e-2, which is why the toy cases are not run that small; the bar itself is not relaxed anywhere.
@pytest.mark.parametrize("cfg_name,B,T", [("tiny", 8, 64), ("tiny3", 2, 136), ("tiny3", 8, 128), ("mid", 2, 64), ("1d_config", 2, 752)])
def test_full_model_fwd_bwd(cuda, cfg_name, B, T):
    cfg, model = load_model(cfg_name, cuda, train=True)
    inp = synth_inputs(cfg, B, T, seed=1, device=cuda)
    xt, ref_pred, ref_loss, ref_grads = to.oracle_train(cfg, model, inp)

    out = model(xt, inp["t"], inp["ids"], inp["mask"]).sample
    assert out.shape == ref_pred.shape and out.dtype == torch.float32
    e_out = rel(out, ref_pred)
    loss = torch.nn.functional.mse_loss(out.float(), inp["noise"].float())
    loss.backward()
    torch.cuda.synchronize()
    assert e_out < TOL, f"output rel err {e_out}"
    named = dict(model.named_parameters())
    worst, missing = [], []
    for k, g_ref in ref_grads.items():
        p = named[k]
        if g_ref is None or g_ref.abs().max() == 0:      # dead proj_out weights never receive a gradient
            assert p.grad is None or p.grad.abs().max() == 0, k
            continue
        if p.grad is None:
            missing.append(k)
            continue
        worst.append((rel(p.grad, g_ref), k))
    assert not missing, f"no gradient for {missing[:5]}"
    worst.sort(reverse=True)
    # global gradient vector
    gv = torch.cat([named[k].grad.flatten() for _, k in worst])
    gr = torch.cat([ref_grads[k].flatten() for _, k in worst])
    e_all = rel(gv, gr)
    # the reference's own bf16 path (torch.autocast) on the same inputs: the noise floor of bf16 compute at this depth
    ac = to.oracle_train(cfg, model, inp, autocast=True)[3]
    gac = torch.cat([ac[k].flatten() for _, k in worst])
    e_ac = rel(gac, gr)
    print(f"\n[{cfg_name} B={B} T={T}] out {e_out:.2e} grad(all) {e_all:.2e} (reference under torch.autocast(bf16): {e_ac:.2e}) worst {worst[:4]}")
    # north-star: 2e-2 on outputs AND gradients, no escape clause
    assert e_all < TOL, f"global grad rel err {e_all} (reference under autocast: {e_ac})"
    # per-tensor outliers: small tensors deep in the net carry the largest bf16 noise; bound them by the error the
    # reference itself shows when it runs under torch.autocast(bf16) on the same inputs (x3), or 5e-2, whichever is larger
    bad = [(e, k, rel(ac[k], ref_grads[k])) for e, k in worst if e > max(5e-2, 3 * rel(ac[k], ref_grads[k]))]
    assert not bad, f"per-tensor grad rel err out of bounds (ours, name, autocast-ref): {bad[:8]}"


def test_no_grad_inference_matches(cuda):
    cfg, model = load_model("tiny", cuda)
    inp = synth_inputs(cfg, 2, 16, seed=3, device=cuda)
    with torch.no_grad():
        a = model(inp["x0"], inp["t"], inp["ids"], inp["mask"]).sample
        b = model(inp["x0"], int(inp["t"][0]), inp["ids"], inp["mask"], return_dict=False)[0]
    assert a.shape == b.shape and torch.isfinite(a).all()
