"""Algorithmic FLOPs of the denoiser by walking the module tree (SURVEY 8d: the roofline denominator).  Runs on the CPU: only
parameter shapes and the sequence lengths are needed.  Counts 2*M*N*K for every Conv1d / Linear and 4*H*Lq*Lk*d for every
softmax attention; normalisations, activations and the embedding lookup are not counted (they are HBM-bound, see DESIGN.md).

    python tools/count_flops.py [T_frames=752] [L_text=550] [batch=32]
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from torch import nn  # noqa: E402

from prompt_tts_b200.ldm.transformer_1d import Transformer1DModel  # noqa: E402
from prompt_tts_b200.models import TTSSingleSpeaker  # noqa: E402


def conv_flops(m: nn.Conv1d, l_out: int) -> float:
    co, ci, k = m.weight.shape
    return 2.0 * l_out * co * ci * k


def lin_flops(m: nn.Linear, rows: int) -> float:
    return 2.0 * rows * m.weight.shape[0] * m.weight.shape[1]


def block_flops(blk, L: int, Lctx: int, parts=None) -> float:
    """BasicTransformerBlock on L tokens with a context of Lctx tokens.  parts (optional dict): accumulates the cross-attention's
    work on the hidden states ("cross_x": to_q, attention, to_out) and on the context ("cross_kv": to_k, to_v)."""
    f = 0.0
    if parts is not None and blk.attn2 is not None:
        a = blk.attn2
        parts["cross_x"] = parts.get("cross_x", 0.0) + lin_flops(a.to_q, L) + lin_flops(a.to_out[0], L) + 4.0 * L * Lctx * a.inner
        parts["cross_kv"] = parts.get("cross_kv", 0.0) + lin_flops(a.to_k, Lctx) + lin_flops(a.to_v, Lctx)
    for attn, lk, rows_kv in ((blk.attn1, L, L), (blk.attn2, Lctx, Lctx)):
        if attn is None:
            continue
        f += lin_flops(attn.to_q, L) + lin_flops(attn.to_k, rows_kv) + lin_flops(attn.to_v, rows_kv) + lin_flops(attn.to_out[0], L)
        f += 4.0 * L * lk * attn.inner            # QK^T and PV over all heads: 4 * H * L * Lk * d
    f += lin_flops(blk.ff.net[0].proj, L) + lin_flops(blk.ff.net[2], L)
    return f


def resnet_flops(r, L: int) -> float:
    f = conv_flops(r.conv1, L) + conv_flops(r.conv2, L) + lin_flops(r.time_emb_proj, 1)
    if r.conv_shortcut is not None:
        f += conv_flops(r.conv_shortcut, L)
    return f


def transformer1d_flops(t: Transformer1DModel, L: int, Lctx: int, parts=None) -> float:
    return conv_flops(t.proj_in, L) + sum(block_flops(b, L, Lctx, parts) for b in t.transformer_blocks)   # proj_out never runs


def forward_flops(model: TTSSingleSpeaker, T: int, Lt: int, parts=None):
    """Forward FLOPs per sample: (text encoder, UNet).  parts: see block_flops (UNet cross-attention only)."""
    text = sum(block_flops(b, Lt, Lt) for b in model.text_encoder.transformer_blocks)
    u = model.unet
    L = T
    f = conv_flops(u.conv_in, L) + lin_flops(u.time_embedding.linear_1, 1) + lin_flops(u.time_embedding.linear_2, 1)
    for blk in u.down_blocks:
        attns = getattr(blk, "attentions", None)
        for i, r in enumerate(blk.resnets):
            f += resnet_flops(r, L)
            if attns is not None:
                f += transformer1d_flops(attns[i], L, Lt, parts)
        if getattr(blk, "downsamplers", None) is not None:
            L = (L - 1) // 2 + 1
            f += sum(conv_flops(d.conv, L) for d in blk.downsamplers)
    if u.mid_block is not None:
        f += resnet_flops(u.mid_block.resnets[0], L)
        for a, r in zip(u.mid_block.attentions, u.mid_block.resnets[1:]):
            f += transformer1d_flops(a, L, Lt, parts) + resnet_flops(r, L)
    for blk in u.up_blocks:
        attns = getattr(blk, "attentions", None)
        for i, r in enumerate(blk.resnets):
            f += resnet_flops(r, L)
            if attns is not None:
                f += transformer1d_flops(attns[i], L, Lt, parts)
        if getattr(blk, "upsamplers", None) is not None:
            L *= 2
            f += sum(conv_flops(up.conv, L) for up in blk.upsamplers)
    f += conv_flops(u.conv_out, L)
    return text, f


def main():
    T = int(sys.argv[1]) if len(sys.argv) > 1 else 752
    Lt = int(sys.argv[2]) if len(sys.argv) > 2 else 550
    B = int(sys.argv[3]) if len(sys.argv) > 3 else 32
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = json.load(open(os.path.join(root, "configs", "1d_config.json")))
    model = TTSSingleSpeaker(cfg)
    text, unet = forward_flops(model, T, Lt)
    fwd = text + unet
    print(f"forward per sample: text {text / 1e9:.1f} GFLOP + UNet {unet / 1e9:.1f} GFLOP = {fwd / 1e9:.1f} GFLOP")
    print(f"forward + backward (3x): {3 * fwd / 1e9:.1f} GFLOP / sample = {3 * fwd / T / 1e9:.3f} GFLOP / frame")
    print(f"train step, batch {B}: {3 * fwd * B / 1e12:.2f} TFLOP;  at 1391 TFLOP/s sustained: {3 * fwd * B / 1391e12 * 1e3:.1f} ms")
    print(f"sampling, 100 steps: {(text + 100 * unet) / 1e12:.2f} TFLOP / utterance")
    parts = {}
    forward_flops(model, T, Lt, parts)
    step = unet - parts["cross_kv"]       # a sampling step: the context's K / V are projected once per sample() call
    guided = 2 * step - parts["cross_x"]  # classifier-free guidance: the null-context rows skip to_q, attention and to_out
    print(f"sampling step per sample: {step / 1e9:.1f} GFLOP (cross-attention on x: {parts['cross_x'] / 1e9:.1f}); guided "
          f"(2 rows, null-context cross-attention skipped): {guided / 1e9:.1f} GFLOP = {guided / step:.3f} x unguided")


if __name__ == "__main__":
    main()
