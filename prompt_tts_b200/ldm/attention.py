"""Parameter holders + tape forward for the diffusers-0.15 pieces the reference imports
(`BasicTransformerBlock`, `Attention`, `FeedForward`/`GEGLU`, `Timesteps`, `TimestepEmbedding`;
import sites: reference tts/ldm/transformer_1d.py:11, tts/models.py:8, tts/ldm/unet_1d_condition.py:21).

The `nn.Linear` / `nn.LayerNorm` children exist only to own parameters under the reference's state_dict names
(and to draw the same default initialisation in the same order); their `forward` is never called -- all
arithmetic goes through `prompt_tts_b200.engine` (hand-written sm_100a kernels).
"""
from __future__ import annotations

import torch
from torch import nn

from .. import engine as E
from .. import ops


class Attention(nn.Module):
    """diffusers Attention: to_q/to_k/to_v without bias, to_out = [Linear(bias), Dropout], scale 1/sqrt(dim_head)."""

    def __init__(self, query_dim, cross_attention_dim=None, heads=8, dim_head=64, dropout=0.0, bias=False, upcast_attention=False):
        super().__init__()
        inner = heads * dim_head
        self.heads, self.dim_head, self.inner = heads, dim_head, inner
        self.is_cross = cross_attention_dim is not None
        ctx = cross_attention_dim if cross_attention_dim is not None else query_dim
        self.scale = dim_head ** -0.5
        assert not bias, "the reference path builds q/k/v without bias"
        self.to_q = nn.Linear(query_dim, inner, bias=False)
        self.to_k = nn.Linear(ctx, inner, bias=False)
        self.to_v = nn.Linear(ctx, inner, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(inner, query_dim), nn.Dropout(dropout)])

    def _fwd(self, tape, hn: E.Var, ctx, residual: E.Var, out=None) -> E.Var:
        """hn: normed hidden states [B, L, C]; ctx: encoder states Var [B, Lk, Cctx] or None (self-attention).
        out: optional destination of the result (E.linear)."""
        C = self.inner
        if ctx is None:
            qkv = E.linear(tape, hn, [self.to_q.weight, self.to_k.weight, self.to_v.weight])      # fused QKV GEMM
            o = E.attention_core(tape, qkv, 0, qkv, C, 2 * C, self.heads, C)
        elif id(self) in tape.kv_group:
            # this layer's K / V are columns of the grouped projection computed once per forward (Unet1DConditionModel._fwd)
            q = E.linear(tape, hn, [self.to_q.weight])
            kv_all, k_off, v_off = tape.kv_group[id(self)]
            o = E.attention_core(tape, q, 0, kv_all, k_off, v_off, self.heads, C, shared_kv=True)
        else:
            q = E.linear(tape, hn, [self.to_q.weight])
            kv = None if tape.kv_cache is None or tape.recording else tape.kv_cache.get(id(self))
            if kv is None:
                kv = E.linear(tape, ctx, [self.to_k.weight, self.to_v.weight])                    # fused KV GEMM
                if tape.kv_cache is not None and not tape.recording:
                    tape.kv_cache[id(self)] = kv
            o = E.attention_core(tape, q, 0, kv, 0, C, self.heads, C)
        return E.linear(tape, o, [self.to_out[0].weight], [self.to_out[0].bias], residual=residual, out=out)


class GEGLU(nn.Module):
    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)


class FeedForward(nn.Module):
    def __init__(self, dim, mult=4, dropout=0.0):
        super().__init__()
        inner = int(dim * mult)
        self.net = nn.ModuleList([GEGLU(dim, inner), nn.Dropout(dropout), nn.Linear(inner, dim)])

    def _fwd(self, tape, hn: E.Var, residual: E.Var) -> E.Var:
        u = E.linear(tape, hn, [self.net[0].proj.weight], [self.net[0].proj.bias])
        g = E.geglu(tape, u)
        return E.linear(tape, g, [self.net[2].weight], [self.net[2].bias], residual=residual)


class BasicTransformerBlock(nn.Module):
    """Pre-LN block: h += attn1(LN1 h); h += attn2(LN2 h, enc) (only when built with cross_attention_dim);
    h += FF(LN3 h).  Construction order follows diffusers so seeded initialisation matches."""

    def __init__(self, dim, num_attention_heads, attention_head_dim, dropout=0.0, cross_attention_dim=None,
                 activation_fn="geglu", num_embeds_ada_norm=None, attention_bias=False, only_cross_attention=False,
                 upcast_attention=False, norm_elementwise_affine=True, norm_type="layer_norm", final_dropout=False):
        super().__init__()
        assert activation_fn == "geglu" and norm_type == "layer_norm" and num_embeds_ada_norm is None and not only_cross_attention
        assert dropout == 0.0, "the reference path runs with dropout 0"
        self.attn1 = Attention(dim, None, num_attention_heads, attention_head_dim, dropout, attention_bias)
        self.ff = FeedForward(dim, dropout=dropout)
        if cross_attention_dim is not None:
            self.attn2 = Attention(dim, cross_attention_dim, num_attention_heads, attention_head_dim, dropout, attention_bias)
            self.norm2 = nn.LayerNorm(dim)
        else:
            self.attn2 = None
            self.norm2 = None
        self.norm1 = nn.LayerNorm(dim)
        self.norm3 = nn.LayerNorm(dim)

    def _fwd(self, tape, h: E.Var, enc) -> E.Var:
        n = E.layernorm(tape, h, self.norm1.weight, self.norm1.bias)
        h = self.attn1._fwd(tape, n, None, h)
        if self.attn2 is not None:
            if tape.cond_rows is not None:
                h = self._cross_guided(tape, h, enc)
            else:
                n = E.layernorm(tape, h, self.norm2.weight, self.norm2.bias)
                h = self.attn2._fwd(tape, n, enc, h)
        n = E.layernorm(tape, h, self.norm3.weight, self.norm3.bias)
        return self.ff._fwd(tape, n, h)

    def _cross_guided(self, tape, h: E.Var, enc) -> E.Var:
        """h += attn2(LN2 h, ctx) for a classifier-free-guidance batch (inference only): rows [0, Bc) of h (Bc = tape.cond_rows)
        attend to `enc` [Bc, Lk, Cctx]; the rows after them have the null context, an all-zero one.  For those, K = V = 0 (to_k and
        to_v have no bias), the softmax weights are uniform and P V = 0, so to_out's GEMM sees a zero operand and its epilogue
        writes bf16(h + bias): that is computed directly (pt_rows_add_bias_bf16), with no K / V, attention or GEMM for those rows.
        LN2, to_q, the attention and to_out run on the conditional row prefix only, to_out writing into the prefix of the output."""
        assert not tape.recording, "the null-context shortcut of guided sampling is inference-only"
        Bc = tape.cond_rows
        hd = h.data
        Bt, L, C = hd.shape
        assert 0 < Bc < Bt and enc.data.shape[0] == Bc, (Bc, Bt, tuple(enc.data.shape))
        out = torch.empty_like(hd)
        hc = E.Var(hd[:Bc], needs_grad=False)
        n = E.layernorm(tape, hc, self.norm2.weight, self.norm2.bias)
        self.attn2._fwd(tape, n, enc, hc, out=out[:Bc])
        ops.call("rows_add_bias_bf16", ops._p(hd[Bc:]), ops._p(self.attn2.to_out[0].bias.detach()), ops._p(out[Bc:]),
                 (Bt - Bc) * L, C, ops._stream())
        return E.Var(out)


class Timesteps(nn.Module):
    def __init__(self, num_channels, flip_sin_to_cos, downscale_freq_shift):
        super().__init__()
        assert flip_sin_to_cos and downscale_freq_shift == 0, "only the configuration the reference uses"
        self.num_channels = num_channels


class TimestepEmbedding(nn.Module):
    def __init__(self, in_channels, time_embed_dim, act_fn="silu", out_dim=None, post_act_fn=None, cond_proj_dim=None):
        super().__init__()
        assert act_fn == "silu" and post_act_fn is None and cond_proj_dim is None
        self.linear_1 = nn.Linear(in_channels, time_embed_dim)
        self.linear_2 = nn.Linear(time_embed_dim, out_dim if out_dim is not None else time_embed_dim)
