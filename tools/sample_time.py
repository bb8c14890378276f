"""Time one sample() call at the bench's sampling configuration (B = 64, T = 1504, 225-frame prompt).

    python tools/sample_time.py                          # DDPMSampler, 100 steps
    python tools/sample_time.py 20 dpm                   # DPMSolverSampler, 20 steps (samplers: ddpm, ddim, dpm)
    python tools/sample_time.py 100 ddpm 50 ddim 20 dpm --rounds 3    # several configurations, alternating, three rounds
    python tools/sample_time.py 20 dpm --guidance 3 --rounds 3           # each configuration unguided and with guidance_scale 3, alternating

RTF = seconds of GPU time / seconds of audio generated (denoiser only, as bench.py's `sampling` object)."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from prompt_tts_b200.models import TTSSingleSpeaker  # noqa: E402
from prompt_tts_b200.sample import DDIMSampler, DDPMSampler, DPMSolverSampler  # noqa: E402

SAMPLERS = {"ddpm": DDPMSampler, "ddim": DDIMSampler, "dpm": DPMSolverSampler}
B, T, P = 64, 1504, 225

args = sys.argv[1:]
rounds = 1
if "--rounds" in args:
    k = args.index("--rounds")
    rounds = int(args[k + 1])
    del args[k:k + 2]
guidance = None
if "--guidance" in args:
    k = args.index("--guidance")
    guidance = float(args[k + 1])
    del args[k:k + 2]
runs = []
while args:
    steps = int(args.pop(0))
    kind = args.pop(0) if args and not args[0].isdigit() else "ddpm"
    if kind not in SAMPLERS:
        sys.exit(f"unknown sampler {kind!r}: one of {', '.join(SAMPLERS)}")
    runs.append((kind, steps))
runs = runs or [("ddpm", 100)]

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                          text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = "unknown"
print(f"card: {card}")
cfg = bench.load_cfg(bench.CFG)
dev = torch.device("cuda:0")
torch.manual_seed(0)
model = TTSSingleSpeaker(cfg).to(dev).eval()
inp = bench.synth(cfg, B, T, 4000, dev)
prompt = inp["x0"][..., :P].contiguous()
DDPMSampler(model, n_infer=4).sample(inp["ids"], T, prompt=prompt, seed=1)      # untimed: first-use costs (allocator pools, weight packs)
samplers = [(kind, steps, SAMPLERS[kind](model, n_infer=steps)) for kind, steps in runs]
audio_s = B * T / 75.0
scales = [1.0] if guidance is None else [1.0, guidance]
if guidance is not None:      # untimed: first use of the 2B-row shapes
    DDPMSampler(model, n_infer=4).sample(inp["ids"], T, prompt=prompt, seed=1, guidance_scale=guidance)
for r in range(rounds):
    for kind, steps, smp in samplers:
        for w in scales:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            e0.record()
            x = smp.sample(inp["ids"], T, prompt=prompt, seed=0, guidance_scale=w)
            e1.record()
            torch.cuda.synchronize()
            sec = e0.elapsed_time(e1) / 1e3
            peak = torch.cuda.max_memory_allocated() / 2 ** 30
            tag = f" guidance {w:g}" if guidance is not None else ""
            print(f"{kind}{tag} sample(): {sec:.3f} s for {steps} steps ({sec / steps * 1e3:.1f} ms/step), RTF {sec / audio_s:.5f}, "
                  f"peak {peak:.2f} GiB, finite {bool(torch.isfinite(x).all())}" + (f"  [round {r + 1}]" if rounds > 1 else ""))
