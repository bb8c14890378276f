"""Which parameter tensors carry the global gradient error of the B200 path vs the fp32 oracle (tiny configs)."""
import os, sys
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, "tests")); sys.path.insert(0, os.path.join(root, "oracle"))
import torch
from util import load_cfg, rel, synth_inputs
import training_oracle as to
from prompt_tts_b200.models import TTSSingleSpeaker

cfg_name, B, T = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
cuda = torch.device("cuda:0")
cfg = load_cfg(cfg_name)
torch.manual_seed(0)
model = TTSSingleSpeaker(cfg).to(cuda)
inp = synth_inputs(cfg, B, T, seed=1, device=cuda)
xt, ref_pred, ref_loss, ref_grads = to.oracle_train(cfg, model, inp)
out = model(xt, inp["t"], inp["ids"], inp["mask"]).sample
torch.nn.functional.mse_loss(out.float(), inp["noise"].float()).backward()
ac = to.oracle_train(cfg, model, inp, autocast=True)[3]
named = dict(model.named_parameters())
rows = []
tot_e = tot_r = tot_a = 0.0
for k, g in ref_grads.items():
    p = named[k]
    if g is None or p.grad is None or g.abs().max() == 0:
        continue
    e = (p.grad - g).pow(2).sum().item(); r = g.pow(2).sum().item(); a = (ac[k] - g).pow(2).sum().item()
    rows.append((e, r, a, k)); tot_e += e; tot_r += r; tot_a += a
print(f"global: ours {(tot_e/tot_r)**.5:.3e}  autocast-ref {(tot_a/tot_r)**.5:.3e}  out {rel(out, ref_pred):.3e}")
rows.sort(reverse=True)
for e, r, a, k in rows[:25]:
    print(f"{100*e/tot_e:5.1f}% of err  ours {(e/r)**.5:.2e}  autocast {(a/r)**.5:.2e}  |g|^2 share {100*r/tot_r:5.1f}%  {k}")
