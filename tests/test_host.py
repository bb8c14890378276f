"""CPU: host-side logic -- the C ABI library loads and exports every declared symbol, the drop-in module tree has the
reference's state_dict, the product refuses to run without a GPU, and the data-parallel bucket logic (gloo, world 2)."""
import os
import re
import subprocess
import sys

import pytest
import torch

from util import ROOT, load_cfg


def test_abi_exports_every_declared_symbol():
    from prompt_tts_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "prompt_tts_b200.h")).read()
    declared = set(re.findall(r"\b(pt_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 40
    l = _lib.lib()
    for name in sorted(declared):
        assert hasattr(l, name), f"{name} declared in the header but not exported by libpt_b200.so"
    assert l.pt_version() >= 1
    for name in _lib.EXPORTS:
        assert name in declared, f"{name} bound in _lib.py but missing from the header"


def test_state_dict_matches_reference_layout():
    import ref_model
    from prompt_tts_b200.models import TTSSingleSpeaker
    for name in ["tiny", "tiny3"]:
        cfg = load_cfg(name)
        m = TTSSingleSpeaker(cfg)
        sd = m.state_dict()
        shapes = ref_model.param_shapes(cfg)
        assert set(sd.keys()) == set(shapes.keys())
        for k, v in sd.items():
            assert tuple(v.shape) == tuple(shapes[k]), k
        m.load_state_dict(ref_model.random_state_dict(cfg, 0), strict=True)
    with torch.device("meta"):
        full = TTSSingleSpeaker(load_cfg("1d_config"))
    assert len(full.state_dict()) == 740
    assert sum(p.numel() for p in full.parameters()) == 536_767_432


def test_product_fails_loudly_without_gpu():
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.models import TTSSingleSpeaker
    cfg = load_cfg("tiny")
    m = TTSSingleSpeaker(cfg)
    x = torch.zeros(1, 8, 16)
    with pytest.raises(_lib.PtError):
        m(x, 3, torch.zeros(1, 24, dtype=torch.int32), None)


def test_sampler_and_optimizer_fail_loudly():
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.models import TTSSingleSpeaker
    from prompt_tts_b200.optim import FusedClipAdamW
    from prompt_tts_b200.sample import DDPMSampler
    from prompt_tts_b200.train import DenoiserTrainStep
    m = TTSSingleSpeaker(load_cfg("tiny"))
    with pytest.raises(_lib.PtError):                      # CPU tensors: there is no CPU fallback
        DDPMSampler(m, n_infer=2).sample(torch.zeros(1, 24, dtype=torch.int32), 16)
    with pytest.raises(_lib.PtError):                      # the flat gradient layout is defined by the first train step
        FusedClipAdamW(DenoiserTrainStep(m)).step()
    smp = DDPMSampler(m, n_infer=100)
    assert smp.timesteps[0] == 990 and smp.timesteps[-1] == 0 and len(smp.timesteps) == 100     # set_timesteps(100) over 1000


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "prompt_tts_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                code = "\n".join(l for l in src.splitlines() if not l.lstrip().startswith(("//", "#", "*", "/*")))
                assert not re.search(r"(import|from|include|dlopen|CDLL)[^\n]*(ref_model|rvq_oracle|seanet_oracle|seanet_emul|oracle[/.])", code), f


def test_gradsync_gloo_world2():
    """Two CPU ranks over gloo drive GradSync with the real tape's gradient bookkeeping (plain, stacked and tap-major conv groups):
    parameters are broadcast from rank 0, every step both ranks hold the mean, micro-steps without sync accumulate locally and
    the last one reduces the window's sum, and a changed completion order is refused."""
    code = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from prompt_tts_b200.dp import GradSync
from prompt_tts_b200.engine import Tape, PackCache
rank = int(os.environ["RANK"])
dist.init_process_group("gloo", rank=rank, world_size=2)
torch.manual_seed(rank)
model = torch.nn.Module()
model.a = torch.nn.Parameter(torch.randn(1000)); model.b = torch.nn.Parameter(torch.randn(30, 100))
model.q = torch.nn.Parameter(torch.randn(16, 8)); model.k = torch.nn.Parameter(torch.randn(24, 8))
model.c = torch.nn.Parameter(torch.randn(12, 10, 3)); model.d = torch.nn.Parameter(torch.randn(70001))
gs = GradSync(model, world_size=2, bucket_mb=0.01)
ref = [torch.zeros(1)]
dist.broadcast(ref[0], 0)
chk = model.a.detach().clone(); dist.broadcast(chk, 0)
assert torch.equal(chk, model.a.detach()), "parameters must be broadcast from rank 0 at construction"
for step in range(3):
    tape = Tape(PackCache()); gs.attach(tape)
    done = 0
    for i, get in enumerate([lambda: tape.pgrad(model.a), lambda: tape.pgrad(model.b), lambda: tape.pgrad_cat([model.q, model.k]),
                             lambda: tape.pgrad_conv(model.c), lambda: tape.pgrad(model.d)]):
        buf = get(); buf += float((rank + 1) * (i + 1) * (step + 1))
        if tape.on_ready and len(tape.pgrad_order) > done:
            tape.on_ready(tape.pgrad_order[done:]); done = len(tape.pgrad_order)
    gs.finish()
    for i, p in enumerate([model.a, model.b, model.q, model.c, model.d]):
        g = tape.pgrads[id(p)]
        assert g.shape == p.shape
        want = 1.5 * (i + 1) * (step + 1)
        assert torch.allclose(g, torch.full_like(g, want)), (step, i, g.flatten()[:3], want)
        assert g.untyped_storage().data_ptr() == gs.flat.untyped_storage().data_ptr(), "param.grad must be a view of the flat buffer from step 1 on"
    assert tape.pgrads[id(model.k)].shape == model.k.shape and not tape.pgrads[id(model.c)].is_contiguous()
    if step > 0: assert gs.n_buckets_last > 1
# accumulation window of two micro-steps: no exchange in the first, the sum is reduced in the second
for micro in range(2):
    tape = Tape(PackCache()); gs.attach(tape, zero=micro == 0, sync=micro == 1)
    done = 0
    for i, get in enumerate([lambda: tape.pgrad(model.a), lambda: tape.pgrad(model.b), lambda: tape.pgrad_cat([model.q, model.k]),
                             lambda: tape.pgrad_conv(model.c), lambda: tape.pgrad(model.d)]):
        buf = get(); buf += float(rank + 1)
        tape.on_ready(tape.pgrad_order[done:]); done = len(tape.pgrad_order)
    gs.finish()
    want = float(rank + 1) if micro == 0 else 3.0
    assert torch.allclose(tape.pgrads[id(model.d)], torch.full((70001,), want)), (micro, tape.pgrads[id(model.d)][:3])
# a different completion order is an error, not a silently wrong bucket
tape = Tape(PackCache()); gs.attach(tape)
tape.pgrad(model.b)
try:
    tape.on_ready(tape.pgrad_order[0:]); bad = False
except RuntimeError:
    bad = True
assert bad
dist.destroy_process_group()
print("OK", rank)
''' % ROOT
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29531")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "OK" in o, o[-2000:]


def test_codec_leg_collectives_gloo_world2():
    """bench.py's codec leg with two CPU ranks over gloo and a stubbed local measurement: the two max-over-ranks reductions run on
    every rank whatever happened locally -- a rank whose kernels failed must not leave the other one waiting in an all-reduce --
    and the line carries the slowest rank's time."""
    code = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
import bench
rank = int(os.environ["RANK"])
dist.init_process_group("gloo", rank=rank, world_size=2)
def mx(x):
    t = torch.tensor([x], dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t.item())
bench._codec_local = lambda dev, torch_, rank_, B, secs: (0.10 + 0.05 * rank_, 0.20 - 0.05 * rank_, 24, 24, True)
line = bench.codec_throughput("cpu", torch, rank, 2, mx)
assert abs(line["encode_ms"] - 150.0) < 1e-6 and abs(line["decode_ms"] - 200.0) < 1e-6 and line["n_gpus"] == 2, line
assert abs(line["encode_audio_s_per_s"] - 2 * 32 * 12 / 0.15) < 1e-6
assert abs(line["roofline"]["peak_tflops"] / 2 - 72.49) < 0.5
def boom(*a):
    if a[2] == 1: raise RuntimeError("kernel failed on this rank")
    return (0.1, 0.2, 24, 24, True)
bench._codec_local = boom
line = bench.codec_throughput("cpu", torch, rank, 2, mx)
assert "unavailable" in line and (("kernel failed" in line["unavailable"]) == (rank == 1)), line
dist.destroy_process_group()
print("OK", rank)
''' % ROOT
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "OK" in o, o[-2000:]


def test_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) emits exactly one JSON line on stdout with
    the contract's keys, runs on the host cores only and reports itself as the oracle port."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "denoiser_train_codec_frames_per_sec" and d["unit"] == "frames/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: the loss, a gradient sample taken at the same positions every time (in the parameters' logical
    element order, whatever the layout of the gradient view) and every gradient's norm, as float32 / float64 .npy files within the
    64 MB a dump may take; --steps below one and a dump of the CPU arm are refused."""
    import numpy as np
    import bench
    assert bench.DUMP_GRAD_SAMPLE * 4 + 4096 * 8 <= 64 << 20
    monkeypatch.setattr(bench, "DUMP_GRAD_SAMPLE", 16)
    m = torch.nn.Module()
    m.a, m.dead, m.b = (torch.nn.Parameter(torch.zeros(s)) for s in ((5, 7), (3,), (11,)))
    m.a.grad = torch.arange(35.0).reshape(5, 7).t().contiguous().t()      # a non-contiguous view, like a k=3 conv weight's gradient
    m.b.grad = torch.arange(11.0) + 100
    values = set(range(35)) | set(range(100, 111))
    dumps = []
    for d in (tmp_path / "one", tmp_path / "two"):
        bench.dump_outputs(str(d), m, torch.tensor(0.25), torch)
        got = {n: np.load(d / f"{n}.npy") for n in ("loss", "grad_sample", "grad_norms")}
        assert got["loss"].dtype == np.float32 and got["loss"].shape == () and got["loss"] == 0.25
        assert got["grad_norms"].dtype == np.float64 and np.allclose(got["grad_norms"], [m.a.grad.norm(), m.b.grad.norm()])
        s = got["grad_sample"]
        assert s.dtype == np.float32 and s.shape == (16,) and set(s.tolist()) <= values and (np.diff(s) >= 0).all()
        dumps.append(s)
    assert np.array_equal(dumps[0], dumps[1])
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr, (argv, r.stderr[-500:])


def test_flop_count_matches_the_survey():
    """tools/count_flops.py walks the module tree of the full config: the roofline denominators of SURVEY 8(d)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import count_flops
    from prompt_tts_b200.models import TTSSingleSpeaker
    model = TTSSingleSpeaker(load_cfg("1d_config"))
    text, unet = count_flops.forward_flops(model, 752, 550)
    assert abs(text / 1e9 - 45.2) < 0.1 and abs(unet / 1e9 - 218.2) < 0.1          # 263.4 GFLOP forward per sample
    assert abs(3 * (text + unet) * 32 / 1e12 - 25.29) < 0.01                       # one train step at batch 32
    text2, unet2 = count_flops.forward_flops(model, 1504, 550)
    assert abs(unet2 / 1e9 - 428.0) < 0.1 and abs((text2 + 100 * unet2) / 1e12 - 42.84) < 0.01   # sampling, per utterance


def test_conv_tile_choice_and_gemm_tile_table():
    """Host logic that needs no GPU: which k=3 convolutions run with the weights on the tile rows (engine._swap_tile), and the
    generated per-shape tile table the library compiles in is well-formed (10 integers per row, a supported tile width)."""
    import re
    from prompt_tts_b200 import engine as E
    assert E._swap_tile(94, 1280) == 96 and E._swap_tile(47, 256) == 64 and E._swap_tile(64, 128) == 64
    assert E._swap_tile(188, 1280) == 0           # two row tiles vs one 192-wide tile: a tie when measured, the old form stays
    assert E._swap_tile(94, 320) == 0             # channel count not a multiple of 128
    assert E._swap_tile(128, 1280) == 0 and E._swap_tile(752, 1280) == 0
    path = os.path.join(ROOT, "prompt_tts_b200", "csrc", "gemm_tile_table.inc")
    rows = [l for l in open(path) if l.strip().startswith("{")]
    assert rows, "empty tile table"
    for l in rows:
        vals = [int(v) for v in re.match(r"\s*\{([^}]*)\}", l).group(1).split(",")]
        assert len(vals) == 10 and vals[0] > 0 and vals[1] > 0 and vals[2] > 0
        assert vals[9] in (64, 128, 160, 192, 224, 256, 257) and vals[5] in (0, 1) and vals[6] in (0, 1) and vals[7] in (0, 2)
