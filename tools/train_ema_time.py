"""Time the bench's full training step (fwd + bwd + clip + AdamW, 1d_config, B = 32, T = 752, one captured CUDA graph per arm)
without and with an EMA of the weights (`optim.FusedEMA`, diffusers' defaults), alternating the arms in one process; also the time
of one `FusedEMA.swapped()` enter + exit and the memory the EMA adds.

    python tools/train_ema_time.py [--steps 20] [--rounds 4]

With the EMA the optimiser step launches one more kernel (the one-thread decay schedule) and its AdamW kernel reads and writes the
fp32 average as well: 8 more bytes per parameter."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from prompt_tts_b200 import _lib  # noqa: E402
from prompt_tts_b200.models import TTSSingleSpeaker  # noqa: E402
from prompt_tts_b200.optim import FusedClipAdamW, FusedEMA  # noqa: E402
from prompt_tts_b200.train import DenoiserTrainStep  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=4)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("train_ema_time.py: needs a CUDA device")
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                          text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = "unknown"
print(f"card: {card}")
dev = torch.device("cuda:0")
cfg = bench.load_cfg(bench.CFG)
B, T = bench.BATCH, bench.T_FRAMES
inp = bench.synth(cfg, B, T, 1000, dev)
lib = _lib.lib()
GB = 1e9


def build(with_ema):
    """One model + stepper + optimiser (+ EMA) per arm: the optimiser re-homes its model's parameters into its own flat buffers."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    torch.manual_seed(0)
    model = TTSSingleSpeaker(cfg).to(dev)
    stepper = DenoiserTrainStep(model)
    opt = FusedClipAdamW(stepper)
    ema = FusedEMA(opt) if with_ema else None
    loss = torch.zeros((), device=dev)

    def step():
        stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"], loss_out=loss)
        opt.step()
    step()                                  # defines the layout; attach() allocates the flat buffers (and the average)
    stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"], loss_out=loss)
    l0 = lib.pt_launch_count()
    opt.step()
    opt_launches = lib.pt_launch_count() - l0
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    g.replay()
    torch.cuda.synchronize()
    mem = (torch.cuda.memory_allocated() - base, torch.cuda.max_memory_allocated() - base)
    return dict(graph=g, opt_launches=opt_launches, mem=mem, keep=(model, stepper, opt, ema, loss))


arms = {"no EMA": build(False), "FusedEMA": build(True)}
for name, a in arms.items():
    print(f"{name}: opt.step() = {a['opt_launches']} launches; resident {a['mem'][0] / GB:.3f} GB, peak {a['mem'][1] / GB:.3f} GB "
          f"above the allocation before the arm was built")
d_res = arms["FusedEMA"]["mem"][0] - arms["no EMA"]["mem"][0]
d_peak = arms["FusedEMA"]["mem"][1] - arms["no EMA"]["mem"][1]
ema = arms["FusedEMA"]["keep"][3]
print(f"EMA adds {d_res / GB:.3f} GB resident, {d_peak / GB:.3f} GB at the peak (average buffer: {ema.eflat.numel() * 4 / GB:.3f} GB, "
      f"{ema.eflat.numel()} fp32 values)")

times = {name: [] for name in arms}
for r in range(args.rounds):
    for name, a in arms.items():
        g = a["graph"]
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        times[name].append(e0.elapsed_time(e1) / args.steps)
        print(f"{name}: {times[name][-1]:.2f} ms/step  [round {r + 1}]")
for name, t in times.items():
    print(f"{name}: median {sorted(t)[len(t) // 2]:.2f} ms/step, min {min(t):.2f}, max {max(t):.2f} over {len(t)} rounds")
print(f"EMA cost (median difference): {sorted(times['FusedEMA'])[len(times['FusedEMA']) // 2] - sorted(times['no EMA'])[len(times['no EMA']) // 2]:+.3f} ms/step")

# the AdamW kernel alone, plain and fused, on each arm's own buffers (fp32 gradients): bytes per element from the kernel's accesses --
# p, m, v read + written (24), g read (4), bf16 shadow written (2); the fused kernel also reads + writes the average (8)
from prompt_tts_b200 import ops  # noqa: E402


def kernel_call(with_ema):
    _, stepper, opt, e, _ = arms["FusedEMA" if with_ema else "no EMA"]["keep"]
    gs = stepper.grad_sync
    if with_ema:
        return lambda: ops.call("adamw_ema_step_dev", ops._p(opt.pflat), ops._p(gs.flat), 0, ops._p(opt.m), ops._p(opt.v),
                                ops._p(opt.wflat), ops._p(e.eflat), gs.total, ops._p(opt.state), ops._p(e.state), ops._stream())
    return lambda: ops.call("adamw_step_dev", ops._p(opt.pflat), ops._p(gs.flat), 0, ops._p(opt.m), ops._p(opt.v), ops._p(opt.wflat),
                            gs.total, ops._p(opt.state), ops._stream())


kt = {False: [], True: []}
for r in range(args.rounds):
    for with_ema in (False, True):
        fn = kernel_call(with_ema)
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        kt[with_ema].append(e0.elapsed_time(e1) / args.steps)
n_el = ema.eflat.numel()
for with_ema, t in kt.items():
    med = sorted(t)[len(t) // 2]
    nbytes = n_el * (38 if with_ema else 30)
    print(f"AdamW kernel {'with EMA' if with_ema else 'plain   '}: median {med:.3f} ms ({min(t):.3f} - {max(t):.3f}), "
          f"{nbytes / GB:.2f} GB -> {nbytes / med / 1e6:.0f} GB/s")

# swapped(): two full passes over master + average + bf16 shadow (10 bytes per parameter each way)
for _ in range(2):
    with ema.swapped():
        pass
n_swap = 10
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(n_swap):
    with ema.swapped():
        pass
e1.record()
torch.cuda.synchronize()
print(f"swapped() enter + exit: {e0.elapsed_time(e1) / n_swap:.3f} ms")
print(f"card: {card}")
