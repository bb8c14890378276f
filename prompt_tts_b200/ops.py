"""Thin Python wrappers over the C ABI (include/prompt_tts_b200.h).  Tensors are torch CUDA tensors used
only as device-memory handles; every computation below is a hand-written sm_100a kernel."""
from __future__ import annotations

import ctypes as C
import math
import numbers
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import Gemm, Operand, Segment, OUT_BF16, OUT_F32, OUT_F32_ATOMIC_ADD, call

BF16 = torch.bfloat16
F32 = torch.float32


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


# diffusers' scheduler `prediction_type` -> PT_PRED_* of the header
PRED_TYPES = {"epsilon": 0, "sample": 1, "v_prediction": 2}


def check_prediction(name: str, prediction_type, snr_gamma=None):
    """Validate a `prediction_type` / `snr_gamma` pair before any device work; returns (PT_PRED_* code, gamma with 0 = off)."""
    if not isinstance(prediction_type, str) or prediction_type not in PRED_TYPES:
        raise ValueError(f"{name}: prediction_type must be one of {sorted(PRED_TYPES)}, got {prediction_type!r}")
    if snr_gamma is not None and (isinstance(snr_gamma, bool) or not isinstance(snr_gamma, numbers.Real)
                                  or not math.isfinite(float(snr_gamma)) or float(snr_gamma) <= 0.0):
        raise ValueError(f"{name}: snr_gamma must be None (no Min-SNR weighting) or a finite real number > 0, got {snr_gamma!r}")
    return PRED_TYPES[prediction_type], (0.0 if snr_gamma is None else float(snr_gamma))


def _need(t: torch.Tensor, dtype, what: str):
    if not t.is_cuda:
        raise _lib.PtError(f"{what}: tensor is not on a CUDA device (no CPU fallback exists)")
    if t.dtype != dtype:
        raise _lib.PtError(f"{what}: expected {dtype}, got {t.dtype}")


# ------------------------------------------------------------------------------------------------ GEMM
def operand(t: torch.Tensor, kmajor: bool, batched: bool = False) -> Operand:
    """`t` is a <=4-D bf16 view in torch order [d3, d2, d1, d0] with d0 contiguous."""
    _need(t, BF16, "gemm operand")
    assert t.dim() <= 4 and t.stride(-1) == 1, (t.shape, t.stride())
    op = Operand()
    op.ptr = t.data_ptr()
    nd = t.dim()
    for i in range(4):
        if i < nd:
            op.dim[i] = t.shape[nd - 1 - i]
            op.stride[i] = t.stride(nd - 1 - i)
        else:
            op.dim[i] = 1
            op.stride[i] = 0
    op.kmajor = 1 if kmajor else 0
    op.batched = 1 if batched else 0
    return op


def segment(nk, a_idx=0, b_idx=0, a_k0=0, b_k0=0, a_shift=0, b_shift=0, nrep=1, rep_is_batch=False, rep_c2_0=0, b_k0_z2=0) -> Segment:
    s = Segment()
    s.b_k0_z2 = b_k0_z2
    s.a_idx, s.b_idx, s.a_k0, s.b_k0 = a_idx, b_idx, a_k0, b_k0
    s.a_mn_shift, s.b_mn_shift, s.nk, s.nrep = a_shift, b_shift, nk, nrep
    s.rep_is_batch, s.rep_c2_0 = (1 if rep_is_batch else 0), rep_c2_0
    return s


def gemm(a: Sequence[Operand], b: Sequence[Operand], segs: Sequence[Segment], M: int, N: int, out: torch.Tensor,
         out_strides=(None, 0, 0), out_mode: int = OUT_BF16, nz2: int = 1, nz3: int = 1, splitk: int = 1,
         alpha: float = 1.0, bias: Optional[torch.Tensor] = None, bias_z2: Optional[torch.Tensor] = None,
         residual: Optional[torch.Tensor] = None, res_strides=(None, 0, 0), block_n: int = 0,
         bias_z2_stride: int = 0, out_stride_n: int = 0, out_transposed: bool = False) -> None:
    """out[z2, z3, m, n] (element strides out_strides = (m, z2, z3)) = epilogue(sum over segments).
    out_transposed (bf16 only): out / residual are [z2, z3, n, m] (m contiguous, out_strides[0] = stride of n), bias / bias_z2 per m."""
    g = Gemm()
    for i, o in enumerate(a):
        g.a[i] = o
    for i, o in enumerate(b):
        g.b[i] = o
    for i, s in enumerate(segs):
        g.seg[i] = s
    g.nseg = len(segs)
    g.M, g.N, g.nz2, g.nz3, g.splitk, g.block_n = M, N, nz2, nz3, splitk, block_n
    g.out = out.data_ptr()
    g.out_dtype = out_mode
    if out_mode == OUT_BF16:
        _need(out, BF16, "gemm out")
    else:
        _need(out, F32, "gemm out")
    g.out_stride_m = out_strides[0] if out_strides[0] is not None else N
    g.out_stride_z2, g.out_stride_z3 = out_strides[1], out_strides[2]
    g.alpha = alpha
    g.out_stride_n = out_stride_n
    g.out_transposed = 1 if out_transposed else 0
    if bias is not None:
        _need(bias, F32, "gemm bias")
        g.bias = bias.data_ptr()
    if bias_z2 is not None:
        _need(bias_z2, F32, "gemm bias_z2")
        g.bias_z2 = bias_z2.data_ptr()
        g.bias_z2_stride = bias_z2_stride
    if residual is not None:
        _need(residual, BF16, "gemm residual")
        g.residual = residual.data_ptr()
        g.res_stride_m = res_strides[0] if res_strides[0] is not None else N
        g.res_stride_z2, g.res_stride_z3 = res_strides[1], res_strides[2]
    call("gemm", C.byref(g), _stream())


# ------------------------------------------------------------------------------------------------ thin wrappers
def empty(shape, dtype=BF16, like: Optional[torch.Tensor] = None, device=None):
    return torch.empty(shape, dtype=dtype, device=(like.device if like is not None else device))


def groupnorm_stats(x: torch.Tensor, G: int, eps: float) -> torch.Tensor:
    B, L, Cc = x.shape
    stats = torch.empty(B, G, 2, dtype=F32, device=x.device)
    call("groupnorm_stats", _p(x), _p(stats), B, L, Cc, G, eps, _stream())
    return stats


def groupnorm_apply(x, stats, gamma, beta, G: int, act: bool) -> torch.Tensor:
    B, L, Cc = x.shape
    y = torch.empty_like(x)
    call("groupnorm_apply", _p(x), _p(stats), _p(gamma), _p(beta), _p(y), B, L, Cc, G, 1 if act else 0, _stream())
    return y


def groupnorm_fwd(x, gamma, beta, G: int, eps: float, act: bool):
    """(y, stats): statistics and normalisation (+ SiLU) in one call -- one read of x when a sample fits in a cluster's shared memory."""
    B, L, Cc = x.shape
    y = torch.empty_like(x)
    stats = torch.empty(B, G, 2, dtype=F32, device=x.device)
    call("groupnorm_fwd", _p(x), _p(gamma), _p(beta), _p(y), _p(stats), B, L, Cc, G, eps, 1 if act else 0, _stream())
    return y, stats


def groupnorm_bwd(dy, x, stats, gamma, beta, dgamma, dbeta, G: int, act: bool, dx_add=None, out=None) -> torch.Tensor:
    """dx (+ dx_add: the gradient that already reached x through another branch, fused into the same pass; `out` may be dx_add)."""
    B, L, Cc = x.shape
    dx = torch.empty_like(x) if out is None else out
    scratch = torch.empty(B, G, 2, dtype=F32, device=x.device)
    call("groupnorm_bwd", _p(dy), _p(x), _p(stats), _p(gamma), _p(beta), _p(dx_add), _p(dx), _p(dgamma), _p(dbeta), _p(scratch),
         B, L, Cc, G, 1 if act else 0, _stream())
    return dx


def layernorm_fwd(x2d, gamma, beta, eps=1e-5):
    M, Cc = x2d.shape
    y = torch.empty_like(x2d)
    rs = torch.empty(M, 2, dtype=F32, device=x2d.device)
    call("layernorm_fwd", _p(x2d), _p(gamma), _p(beta), _p(y), _p(rs), M, Cc, eps, _stream())
    return y, rs


def layernorm_bwd(dy, x2d, rs, gamma, dgamma, dbeta, dx_add=None):
    M, Cc = x2d.shape
    dx = torch.empty_like(x2d)
    call("layernorm_bwd", _p(dy), _p(x2d), _p(rs), _p(gamma), _p(dx_add), _p(dx), _p(dgamma), _p(dbeta), M, Cc, _stream())
    return dx


def softmax_fwd(S, P, rows, n, ld):
    call("softmax_fwd", _p(S), _p(P), rows, n, ld, ld, _stream())


def softmax_bwd(dP, P, dS, rows, n, ld, scale):
    call("softmax_bwd", _p(dP), _p(P), _p(dS), rows, n, ld, ld, scale, _stream())


def _attn_desc(q, k, v, o, lse, heads: int, d: int, scale: float) -> "_lib.Attn":
    """q [B, Lq, >=H*d] / k, v [B, Lk, >=H*d] / o [B, Lq, >=H*d]: bf16 column-slice views (last stride 1)."""
    a = _lib.Attn()
    for t, what in ((q, "q"), (k, "k"), (v, "v"), (o, "o")):
        _need(t, BF16, "attention " + what)
        assert t.dim() == 3 and t.stride(2) == 1, (what, t.shape, t.stride())
    assert k.stride() == v.stride() and k.shape == v.shape
    _need(lse, F32, "attention lse")
    B, Lq, _ = q.shape
    a.q, a.q_rs, a.q_bs = q.data_ptr(), q.stride(1), q.stride(0)
    a.k, a.v, a.kv_rs, a.kv_bs = k.data_ptr(), v.data_ptr(), k.stride(1), k.stride(0)
    a.o, a.o_rs, a.o_bs = o.data_ptr(), o.stride(1), o.stride(0)
    a.lse = lse.data_ptr()
    a.B, a.H, a.Lq, a.Lk, a.d, a.scale = B, heads, Lq, k.shape[1], d, scale
    return a


def attn_fwd(q, k, v, o, lse, heads: int, d: int, scale: float) -> None:
    """o = softmax(q k^T * scale) v per head, lse[B, H, Lq] = log-sum-exp of the scaled logits (fused tcgen05 kernel)."""
    a = _attn_desc(q, k, v, o, lse, heads, d, scale)
    call("attn_fwd", C.byref(a), _stream())


def attn_bwd(q, k, v, o, lse, d_o, dq, dk, dv, heads: int, d: int, scale: float) -> None:
    """dq, dk, dv (column-slice views like q, k, v) from d_o; the logits are recomputed from q, k and lse."""
    a = _attn_desc(q, k, v, o, lse, heads, d, scale)
    for t, what in ((d_o, "d_o"), (dq, "dq"), (dk, "dk"), (dv, "dv")):
        _need(t, BF16, "attention " + what)
        assert t.dim() == 3 and t.stride(2) == 1, (what, t.shape, t.stride())
    assert dk.stride() == dv.stride()
    delta = torch.empty_like(lse)
    a.d_o, a.do_rs, a.do_bs = d_o.data_ptr(), d_o.stride(1), d_o.stride(0)
    a.dq, a.dq_rs, a.dq_bs = dq.data_ptr(), dq.stride(1), dq.stride(0)
    a.dk, a.dv, a.dkv_rs, a.dkv_bs = dk.data_ptr(), dv.data_ptr(), dk.stride(1), dk.stride(0)
    a.delta = delta.data_ptr()
    call("attn_bwd", C.byref(a), _stream())


def geglu_fwd(u2d):
    M, F2 = u2d.shape
    y = torch.empty(M, F2 // 2, dtype=BF16, device=u2d.device)
    call("geglu_fwd", _p(u2d), _p(y), M, F2 // 2, _stream())
    return y


def geglu_bwd(dy, u2d):
    M, F2 = u2d.shape
    du = torch.empty_like(u2d)
    call("geglu_bwd", _p(dy), _p(u2d), _p(du), M, F2 // 2, _stream())
    return du


def add_(a, b, out=None):
    """out = a + b (bf16, same shape, contiguous); out may alias a or b."""
    out = torch.empty_like(a) if out is None else out
    call("add_bf16", _p(a), _p(b), _p(out), a.numel(), _stream())
    return out


def copy2d(src, ld_src, dst, ld_dst, rows, cols):
    call("copy2d_bf16", _p(src), ld_src, _p(dst), ld_dst, rows, cols, _stream())


def upsample2_fwd(x):
    B, L, Cc = x.shape
    y = torch.empty(B, 2 * L, Cc, dtype=BF16, device=x.device)
    call("upsample2_fwd", _p(x), _p(y), B, L, Cc, _stream())
    return y


def upsample2_bwd(dy):
    B, L2, Cc = dy.shape
    dx = torch.empty(B, L2 // 2, Cc, dtype=BF16, device=dy.device)
    call("upsample2_bwd", _p(dy), _p(dx), B, L2 // 2, Cc, _stream())
    return dx


def ncl_to_nlc(x_ncl):
    B, Cc, L = x_ncl.shape
    y = torch.empty(B, L, Cc, dtype=BF16, device=x_ncl.device)
    call("ncl_f32_to_nlc_bf16", _p(x_ncl), _p(y), B, Cc, L, _stream())
    return y


def nlc_to_ncl(x_nlc):
    B, L, Cc = x_nlc.shape
    y = torch.empty(B, Cc, L, dtype=F32, device=x_nlc.device)
    call("nlc_bf16_to_ncl_f32", _p(x_nlc), _p(y), B, Cc, L, _stream())
    return y


def cast_bf16(x_f32, out=None):
    out = torch.empty(x_f32.shape, dtype=BF16, device=x_f32.device) if out is None else out
    call("cast_f32_to_bf16", _p(x_f32), _p(out), x_f32.numel(), _stream())
    return out


def cast_f32(x_bf16):
    out = torch.empty(x_bf16.shape, dtype=F32, device=x_bf16.device)
    call("cast_bf16_to_f32", _p(x_bf16), _p(out), x_bf16.numel(), _stream())
    return out


def pack_conv_weight(w_f32, out=None):
    Co, Ci, k = w_f32.shape
    out = torch.empty(Co, k * Ci, dtype=BF16, device=w_f32.device) if out is None else out
    call("pack_conv_weight", _p(w_f32), _p(out), Co, Ci, k, _stream())
    return out


def unpack_conv_wgrad(gp, g, accumulate=True):
    Co, Ci, k = g.shape
    call("unpack_conv_wgrad", _p(gp), _p(g), Co, Ci, k, 1 if accumulate else 0, _stream())


def colsum(x2d, out_f32, ld=None, lite=False):
    rows, cols = x2d.shape
    call("colsum_bf16_lite" if lite else "colsum_bf16", _p(x2d), ld if ld is not None else x2d.stride(0), _p(out_f32), rows, cols, _stream())


def batch_colsum(x_blc, out_f32, out_stride):
    B, L, Cc = x_blc.shape
    call("batch_colsum_bf16", _p(x_blc), _p(out_f32), out_stride, B, L, Cc, _stream())


def silu_to_bf16(x_f32):
    y = torch.empty(x_f32.shape, dtype=BF16, device=x_f32.device)
    call("silu_f32_to_bf16", _p(x_f32), _p(y), x_f32.numel(), _stream())
    return y


def silu_bwd(x_f32, dy_f32):
    dx = torch.empty_like(x_f32)
    call("silu_bwd_f32", _p(x_f32), _p(dy_f32), _p(dx), x_f32.numel(), _stream())
    return dx


def time_sinusoid(t_i64, dim):
    out = torch.empty(t_i64.shape[0], dim, dtype=F32, device=t_i64.device)
    call("time_sinusoid", _p(t_i64), _p(out), t_i64.shape[0], dim, _stream())
    return out


class RvqPrepared:
    """Device scratch of the tensor-core quantiser for ONE codebook set: bf16 codebooks, |e|^2, max |e| and the fallback counter.
    Build it once with `rvq_prepare(codebooks)` and pass it to `rvq_encode(..., prepared=...)` to skip the (cheap) per-call
    preparation; it must be rebuilt whenever the codebook values change."""

    def __init__(self, codebooks: torch.Tensor):
        Q, K, D = codebooks.shape
        self.shape = (Q, K, D)
        nbytes = int(_lib.lib().pt_rvq_encode_tc_scratch_bytes(Q, K))
        self.buf = torch.empty(nbytes + 256, dtype=torch.uint8, device=codebooks.device)
        self.off = (-self.buf.data_ptr()) % 256
        self.ready = False

    @property
    def ptr(self) -> C.c_void_p:
        return C.c_void_p(self.buf.data_ptr() + self.off)

    def overflow_frames(self) -> int:
        """Frame-stages that fell back to the exhaustive scan since the last preparation (diagnostic; synchronises)."""
        Q, K, D = self.shape
        o = self.off + Q * K * 4 + 256 + Q * K * D * 2
        return int(self.buf[o:o + 8].view(torch.int64).item())


def rvq_prepare(codebooks: torch.Tensor) -> RvqPrepared:
    _need(codebooks, F32, "rvq_prepare codebooks")
    return RvqPrepared(codebooks.contiguous())


def rvq_encode(latents, codebooks, exhaustive: bool = False, prepared: Optional[RvqPrepared] = None):
    """latents [B, 128, T] fp32, codebooks [Q, K, 128] fp32 -> codes [B, Q, T] int64 (SURVEY R1), bit-identical to the oracle.
    Default: tensor-core pre-selection + exact fp32 re-ranking (csrc/rvq_tc.cu); `exhaustive` (or K not a multiple of 128 / > 1024):
    the exact fp32 search over all codes on the FMA pipe (csrc/rvq.cu).  Both produce the same codes."""
    _need(latents, F32, "rvq_encode latents"); _need(codebooks, F32, "rvq_encode codebooks")
    latents, codebooks = latents.contiguous(), codebooks.contiguous()
    B, D, T = latents.shape
    Q, K, D2 = codebooks.shape
    assert D == D2
    codes = torch.empty(B, Q, T, dtype=torch.int64, device=latents.device)
    if exhaustive or K % 128 != 0 or K > 1024 or D != 128:
        cb_sq = torch.empty(Q, K, dtype=F32, device=latents.device)
        call("rvq_encode_ws", _p(latents), _p(codebooks), _p(cb_sq), _p(codes), B, D, T, Q, K, _stream())
        return codes
    if prepared is None:
        prepared = RvqPrepared(codebooks)
    elif prepared.shape != (Q, K, D):
        raise _lib.PtError(f"rvq_encode: `prepared` was built for codebooks {prepared.shape}, got {(Q, K, D)}")
    prep = 0 if prepared.ready else 1
    call("rvq_encode_tc", _p(latents), _p(codebooks), prepared.ptr, prep, _p(codes), B, D, T, Q, K, _stream())
    prepared.ready = True
    rvq_encode.last_prepared = prepared
    return codes


def rvq_decode(codes, codebooks, gather_l2: bool = False):
    """codes [B, Q, T] int64 -> latents [B, 128, T] fp32 = sum_q E_q[codes_q] (SURVEY R2)."""
    _need(codes, torch.int64, "rvq_decode codes"); _need(codebooks, F32, "rvq_decode codebooks")
    codes, codebooks = codes.contiguous(), codebooks.contiguous()
    B, Q, T = codes.shape
    Q2, K, D = codebooks.shape
    assert Q == Q2
    lat = torch.empty(B, D, T, dtype=F32, device=codes.device)
    if gather_l2:      # round-1 kernel: codebook rows gathered through L2 (kept for A/B measurements and Q*K too large for shared memory)
        call("rvq_decode", _p(codes), _p(codebooks), _p(lat), B, D, T, Q, K, _stream())
    else:
        scratch = torch.empty(B * Q * T, dtype=torch.int16, device=codes.device)
        call("rvq_decode_ws", _p(codes), _p(codebooks), _p(lat), _p(scratch), B, D, T, Q, K, _stream())
    return lat


def codes_affine(codes):
    _need(codes, torch.int64, "codes_affine")
    codes = codes.contiguous()
    x0 = torch.empty(codes.shape, dtype=F32, device=codes.device)
    call("codes_affine", _p(codes), _p(x0), codes.numel(), _stream())
    return x0


def codes_affine_inv(x):
    _need(x, F32, "codes_affine_inv")
    x = x.contiguous()
    c = torch.empty(x.shape, dtype=torch.int64, device=x.device)
    call("codes_affine_inv", _p(x), _p(c), x.numel(), _stream())
    return c
