"""GPU, >= 2 devices: N-rank `GradSync` gradients == single-process gradients of the concatenated batch (SURVEY 4 iii; the reference's
DDP wrap train.py:25-29,67-69 and backward :115).  One process per GPU over NCCL, launched the way the bench is launched.  Skipped on
a single-GPU box (the CPU/gloo variant of the bucket logic is tests/test_host.py::test_gradsync_gloo_world2); the 2-GPU run of this
file is committed as profiles/r02_dp_parity_2gpu.json."""
import json
import os
import subprocess
import sys

import pytest

from util import ROOT

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("cfg,B,T", [("tiny3", 2, 64), ("mid", 2, 64)])
def test_two_rank_gradients_match_single_process(cuda, cfg, B, T):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tests", "dp_worker.py"), cfg, str(B), str(T)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    line = [l for l in r.stdout.splitlines() if l.startswith("DPRESULT ")][-1]
    res = json.loads(line[len("DPRESULT "):])
    print(res)
    # fp32 exchange: identical per-sample arithmetic; only the fp32 summation order of the weight-gradient atomics differs
    assert res["fp32"]["identical_on_all_ranks"] and res["fp32"]["weights_identical_after_step"] and res["fp32"]["buckets"] > 1
    assert res["fp32"]["rel_flat_vs_single_process"] < 1e-5, res
    # bf16 exchange: one bf16 rounding of every averaged gradient element (2^-9 relative)
    assert res["bf16"]["identical_on_all_ranks"] and res["bf16"]["weights_identical_after_step"]
    assert res["bf16"]["rel_flat_vs_single_process"] < 4e-3, res
