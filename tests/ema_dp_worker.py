"""Worker of tests/test_ema_gpu.py::test_two_rank_ema_identical (one process per GPU, launched by torch.distributed.run): every rank
trains 3 steps on its own batch with a `FusedEMA`; the averaged gradients are identical on all ranks, so the weights and the EMA must
be too -- bit for bit, with fp32 and with bf16 gradient exchange."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from util import load_cfg, synth_inputs  # noqa: E402


def main():
    from prompt_tts_b200.dp import GradSync
    from prompt_tts_b200.models import TTSSingleSpeaker
    from prompt_tts_b200.optim import FusedClipAdamW, FusedEMA
    from prompt_tts_b200.train import DenoiserTrainStep
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    cfg_name, B, T = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    cfg = load_cfg(cfg_name)
    out = {"world": world, "cfg": cfg_name, "B_per_rank": B, "T": T}

    def same_everywhere(x):
        gathered = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(gathered, x)
        return all(torch.equal(gathered[0], g) for g in gathered)

    for mode in ("fp32", "bf16"):
        torch.manual_seed(1 + rank)                     # ranks start from DIFFERENT weights: GradSync broadcasts rank 0's
        model = TTSSingleSpeaker(cfg).to(dev)
        gs = GradSync(model, world_size=world, bucket_mb=0.25, comm_dtype=torch.float32 if mode == "fp32" else torch.bfloat16)
        stepper = DenoiserTrainStep(model, grad_sync=gs)
        opt = FusedClipAdamW(stepper, lr=1e-3)
        ema = FusedEMA(opt, decay=0.9)
        inp = synth_inputs(cfg, B, T, seed=100 + rank, device=dev)
        for _ in range(3):
            stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"])
            opt.step()
        torch.cuda.synchronize()
        res = {"optimization_step": ema.optimization_step, "ema_identical_on_all_ranks": same_everywhere(ema.eflat),
               "weights_identical_on_all_ranks": same_everywhere(opt.pflat),
               "ema_moved": not torch.equal(ema.eflat, opt.pflat)}
        if rank == 0:
            out[mode] = res
        del model, stepper, gs, opt, ema
    if rank == 0:
        print("EMARESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
