"""Time the bench training step (fwd + bwd, 1d_config, B = 32, T = 752, one captured CUDA graph) without and with condition
dropout (`DenoiserTrainStep(..., cond_keep=)`, a fresh mask each step), alternating in one process.

    python tools/train_dropout_time.py [--steps 20] [--rounds 3] [--p-uncond 0.1]

Condition dropout adds two launches per step: the selection of the text encoding [B, Lt, 768] bf16 in the forward and of its
gradient in the backward."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from prompt_tts_b200 import _lib  # noqa: E402
from prompt_tts_b200.models import TTSSingleSpeaker  # noqa: E402
from prompt_tts_b200.train import DenoiserTrainStep  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--p-uncond", type=float, default=0.1)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("train_dropout_time.py: needs a CUDA device")
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                          text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = "unknown"
print(f"card: {card}")
dev = torch.device("cuda:0")
cfg = bench.load_cfg(bench.CFG)
torch.manual_seed(0)
model = TTSSingleSpeaker(cfg).to(dev)
B, T = bench.BATCH, bench.T_FRAMES
inp = bench.synth(cfg, B, T, 1000, dev)
loss = torch.zeros((), device=dev)
keep = torch.ones(B, dtype=torch.bool, device=dev)
gen = torch.Generator(device=dev).manual_seed(0)
lib = _lib.lib()


def build(use_keep):
    stepper = DenoiserTrainStep(model)

    def step():
        stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"], loss_out=loss, cond_keep=keep if use_keep else None)
    step()
    l0 = lib.pt_launch_count()
    step()
    launches = lib.pt_launch_count() - l0
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    return g, launches, stepper      # the stepper owns the gradient buffers and schedule tables the graph writes / reads


arms = {"cond_keep=None": build(False), "cond_keep=mask": build(True)}
for name, (_, n, _) in arms.items():
    print(f"{name}: {n} launches per eager step")
for r in range(args.rounds):
    for name, (g, _, _) in arms.items():
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            # a fresh mask per step, written into the captured buffer (what a training loop does); drawn in both arms alike
            torch.ge(torch.rand(B, device=dev, generator=gen), args.p_uncond, out=keep)
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        print(f"{name}: {e0.elapsed_time(e1) / args.steps:.2f} ms/step  [round {r + 1}]")
