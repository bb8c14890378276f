"""B200 drop-in for the reference's tts/models.py: TextEncoder (:73-120), PositionalEncoding1D /
PositionalEncodingPermute1D (:19-70) and TTSSingleSpeaker (:123-172).  `TTSSingleSpeaker(config)` takes the same
config dict, has the same forward signature and the same 740 state_dict entries, so train.py:38,100-105 run
unchanged; one forward = one tape over hand-written sm_100a kernels."""
from __future__ import annotations

from typing import Any, Dict, Optional, Union

import numpy as np
import torch
from torch import nn

from . import engine as E
from . import ops
from .ldm.attention import BasicTransformerBlock
from .ldm.unet_1d_condition import Unet1DConditionModel, UNet1DConditionOutput


class PositionalEncoding1D(nn.Module):
    """Holds the `inv_freq` buffer of the reference (state_dict key text_encoder.pos_embedding.penc.inv_freq)."""

    def __init__(self, channels):
        super().__init__()
        self.org_channels = channels
        channels = int(np.ceil(channels / 2) * 2)
        self.channels = channels
        inv_freq = 1.0 / (10000 ** (torch.arange(0, channels, 2).float() / channels))
        self.register_buffer("inv_freq", inv_freq)
        self.cached_penc = None


class PositionalEncodingPermute1D(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.penc = PositionalEncoding1D(channels)

    @property
    def org_channels(self):
        return self.penc.org_channels

    def table(self, L: int, D: int, device) -> torch.Tensor:
        """pe[l, d] fp32: the reference applies the 1-D encoding to the PERMUTED tensor [B, D, L] (models.py:44-51,64-66),
        so the position index runs over the feature axis d and the frequency index over l:
        pe[l, d] = sin(d * w[l // 2]) for even l, cos(d * w[l // 2]) for odd l.  A constant table, built once per shape."""
        c = self.penc.cached_penc
        if c is not None and c.shape == (L, D) and c.device == device:
            return c
        if L > self.penc.channels:
            raise ValueError(f"text length {L} exceeds cmu_seq_len {self.penc.org_channels}")
        inv_freq = self.penc.inv_freq.detach().to("cpu", torch.float32)
        pos = torch.arange(D, dtype=torch.float32)
        ang = torch.einsum("i,j->ij", pos, inv_freq)                       # [D, channels/2]
        emb = torch.stack((ang.sin(), ang.cos()), dim=-1).flatten(-2, -1)   # [D, channels]
        c = emb[:, :L].t().contiguous().to(device)
        self.penc.cached_penc = c
        return c


class TextEncoder(nn.Module):
    def __init__(self, vocab_len, seq_len, dim, attention_head_dim, dropout=0.0, num_layers=1) -> None:
        super().__init__()
        self.word_embedding = nn.Embedding(vocab_len, dim)
        self.pos_embedding = PositionalEncodingPermute1D(seq_len)
        if dim % attention_head_dim != 0:
            raise ValueError("dim must be a multiple of attention_head_dim")
        num_attention_heads = dim // attention_head_dim
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(dim=dim, num_attention_heads=num_attention_heads, attention_head_dim=attention_head_dim, dropout=dropout)
            for _ in range(num_layers)])

    def _fwd(self, tape, ids_i32: torch.Tensor) -> E.Var:
        B, L = ids_i32.shape
        Wt = self.word_embedding.weight
        V, D = Wt.shape
        pe = self.pos_embedding.table(L, D, ids_i32.device)
        x = torch.empty(B, L, D, dtype=E.BF16, device=ids_i32.device)
        ops.call("text_embed_fwd", ops._p(ids_i32), ops._p(Wt.detach()), ops._p(pe), ops._p(x), B, L, D, V, ops._stream())
        h_emb = E.Var(x)      # distinct name: the closure must not see the rebinding of `h` in the block loop

        def bwd():
            if h_emb.grad is not None:
                ops.call("text_embed_bwd", ops._p(ids_i32), ops._p(h_emb.grad), ops._p(tape.pgrad(Wt)), B, L, D, V, ops._stream())
        tape.record(bwd)
        h = h_emb
        for blk in self.transformer_blocks:
            h = blk._fwd(tape, h, None)      # the mask lands in the unused encoder_hidden_states slot (SURVEY 3.4)
        return h

    def forward(self, input_ids, attention_mask=None):
        if not input_ids.is_cuda:
            raise ops._lib.PtError("TextEncoder: inputs must be CUDA tensors; there is no CPU fallback")
        ids = input_ids.to(torch.int32).contiguous()
        params = [p for p in self.parameters()]

        def runner(tape):
            h = self._fwd(tape, ids)
            out = ops.cast_f32(h.data)

            def seed(gouts):
                h.grad, h.owned = ops.cast_bf16(gouts[0].float().contiguous()), True
            return (out,), seed, lambda: []
        return E.TapeFunction.apply(runner, E.get_cache(self), 0, *params)


class TTSSingleSpeaker(nn.Module):
    def __init__(self, config) -> None:
        super().__init__()
        self.text_encoder = TextEncoder(vocab_len=config["cmu_vocab_len"], seq_len=config["cmu_seq_len"],
                                        dim=config["cross_attention_dim"], attention_head_dim=config["attention_head_dim"],
                                        dropout=config["text_encoder_dropout"], num_layers=config["text_encoder_layers"])
        self.unet = Unet1DConditionModel(sample_size=config["sample_size"], in_channels=config["in_channels"],
                                         out_channels=config["out_channels"], layers_per_block=config["layers_per_block"],
                                         block_out_channels=config["block_out_channels"],
                                         down_block_types=config["down_block_types"], mid_block_type=config["mid_block_type"],
                                         up_block_types=config["up_block_types"], cross_attention_dim=config["cross_attention_dim"])

    def forward(self, sample: torch.FloatTensor, timestep: Union[torch.Tensor, float, int], text_seq_ids: torch.Tensor,
                attention_mask: torch.Tensor, cross_attention_kwargs: Optional[Dict[str, Any]] = None, return_dict: bool = True,
                *, cond_keep: Optional[torch.Tensor] = None):
        """cond_keep (not in the reference): optional bool / uint8 [B] CUDA mask for classifier-free guidance training; samples
        where it is 0 see the null condition (an all-zero text encoding) and send no gradient to the text encoder."""
        if not sample.is_cuda:
            raise ops._lib.PtError("TTSSingleSpeaker: inputs must be CUDA tensors; there is no CPU fallback")
        t = Unet1DConditionModel._timesteps(timestep, sample.shape[0], sample.device)
        keep = E.cond_keep_mask(cond_keep, sample.shape[0], sample.device, "TTSSingleSpeaker") if cond_keep is not None else None
        ids = text_seq_ids.to(device=sample.device, dtype=torch.int32).contiguous()
        params = [p for p in self.parameters()]

        def runner(tape, s):
            enc = self.text_encoder._fwd(tape, ids)
            if keep is not None:
                enc = E.cond_select(tape, enc, keep)
            y, seed = self.unet._fwd(tape, s.detach().float().contiguous(), t, enc)
            return (y,), seed, lambda: [None]

        out = E.TapeFunction.apply(runner, E.get_cache(self), 1, sample, *params)
        if not return_dict:
            return (out,)
        return UNet1DConditionOutput(sample=out)
