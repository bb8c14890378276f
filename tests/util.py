import json
import os

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_cfg(name):
    return json.load(open(os.path.join(ROOT, "configs", name + ".json")))


def load_model(cfg_name, dev, train=False, seed=0):
    """the config and TTSSingleSpeaker(cfg) on dev with the weights torch.manual_seed(seed) draws, in eval mode unless train"""
    from prompt_tts_b200.models import TTSSingleSpeaker
    cfg = load_cfg(cfg_name)
    torch.manual_seed(seed)
    m = TTSSingleSpeaker(cfg).to(dev)
    return cfg, (m if train else m.eval())


def rel(a, b):
    a, b = a.detach().float(), b.detach().float()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def synth_inputs(cfg, B, T, seed=0, device="cpu"):
    """Synthetic batch with the reference's input contract (SURVEY 8a A0 / 8d): codes on the 1024-point grid,
    ids int32 in [1, vocab) with a zero-padded tail, mask = position < len."""
    g = torch.Generator().manual_seed(seed)
    codes = torch.randint(0, 1024, (B, cfg["in_channels"], T), generator=g)
    x0 = (codes.float() / 1023 - 0.5) / 0.5
    noise = torch.randn(B, cfg["in_channels"], T, generator=g)
    t = torch.randint(0, 1000, (B,), generator=g)
    Lt = cfg["cmu_seq_len"]
    ids = torch.randint(1, cfg["cmu_vocab_len"], (B, Lt), generator=g).to(torch.int32)
    lens = torch.randint(max(1, Lt // 5), Lt + 1, (B,), generator=g)
    mask = (torch.arange(Lt)[None, :] < lens[:, None]).to(torch.int32)
    ids = ids * mask
    return dict(x0=x0.to(device), noise=noise.to(device), t=t.to(device), ids=ids.to(device), mask=mask.to(device))
