"""Worker of the two-rank tests (one process per GPU, launched by torch.distributed.run through training_oracle.run_two_ranks), with
fp32 and with bf16 gradient exchange.  `dp_worker.py MODE CFG B T`, MODE:
  grads  (tests/test_dp_gpu.py) N-rank GradSync gradients against a single-process step on the concatenated batch -- the reference's
         DDP contract (train.py:25-29,67-69,100-117);
  ema    (tests/test_ema_gpu.py::test_two_rank_ema_identical) every rank trains 3 steps on its own batch with a `FusedEMA`; the
         averaged gradients are identical on all ranks, so the weights and the EMA must be too -- bit for bit."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from util import load_cfg, rel, synth_inputs  # noqa: E402


def main():
    from prompt_tts_b200.dp import GradSync
    from prompt_tts_b200.models import TTSSingleSpeaker
    from prompt_tts_b200.optim import FusedClipAdamW, FusedEMA
    from prompt_tts_b200.train import DenoiserTrainStep
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    mode, cfg_name, B, T = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4])
    cfg = load_cfg(cfg_name)
    out = {"world": world, "cfg": cfg_name, "B_per_rank": B, "T": T}

    def same_everywhere(x):
        gathered = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(gathered, x)
        return all(torch.equal(gathered[0], g) for g in gathered)

    for comm in ("fp32", "bf16"):
        torch.manual_seed(1 + rank)                     # ranks start from DIFFERENT weights: GradSync must broadcast rank 0's
        model = TTSSingleSpeaker(cfg).to(dev)
        gs = GradSync(model, world_size=world, bucket_mb=0.25, comm_dtype=torch.float32 if comm == "fp32" else torch.bfloat16)
        stepper = DenoiserTrainStep(model, grad_sync=gs)
        inp = synth_inputs(cfg, B, T, seed=100 + rank, device=dev)
        if mode == "grads":
            for _ in range(2):                           # step 1 learns the layout (one blocking reduce); step 2 is the bucketed, overlapped path
                stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
            torch.cuda.synchronize()
            buckets = gs.n_buckets_last
            flat = gs.flat.clone()
            same = same_everywhere(flat)                 # every rank holds the same averaged gradient
            # single process, concatenated batch, same (rank 0) weights
            if rank == 0:
                torch.manual_seed(1)
                ref_model = TTSSingleSpeaker(cfg).to(dev)
                parts = [synth_inputs(cfg, B, T, seed=100 + r, device=dev) for r in range(world)]
                cat = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
                ref = DenoiserTrainStep(ref_model)
                for _ in range(2):
                    ref(cat["x0"], cat["noise"], cat["t"], cat["ids"], cat["mask"])
                torch.cuda.synchronize()
                assert [g[1:] for g in ref.grad_sync.groups] == [g[1:] for g in gs.groups]
                out[comm] = {"rel_flat_vs_single_process": rel(flat, ref.grad_sync.flat), "identical_on_all_ranks": same,
                             "buckets": buckets, "grad_norm": float(flat.norm())}
            # one optimiser step on every rank: weights stay identical across ranks
            opt = FusedClipAdamW(stepper, lr=1e-3)
            opt.step()
            same = same_everywhere(opt.pflat.double().sum().reshape(1))
            if rank == 0:
                out[comm]["weights_identical_after_step"] = same
        else:
            assert mode == "ema", mode
            opt = FusedClipAdamW(stepper, lr=1e-3)
            ema = FusedEMA(opt, decay=0.9)
            for _ in range(3):
                stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
                opt.step()
            torch.cuda.synchronize()
            res = {"optimization_step": ema.optimization_step, "ema_identical_on_all_ranks": same_everywhere(ema.eflat),
                   "weights_identical_on_all_ranks": same_everywhere(opt.pflat), "ema_moved": not torch.equal(ema.eflat, opt.pflat)}
            if rank == 0:
                out[comm] = res
            del ema
        del model, stepper, gs, opt
    if rank == 0:
        print("RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
