"""Tape engine: forward primitives over channels-last bf16 activations, each recording its own backward.

Why a tape and not one torch.autograd.Function per op: the whole denoiser forward+backward is ~2.5k kernel
launches; a hand-rolled tape keeps the host cost per launch at one ctypes call, lets backward kernels fuse
gradient accumulation into GEMM epilogues, and is capturable in a CUDA graph.  The tape is bridged to
torch.autograd once per public `forward` (see `TapeFunction`), so `loss.backward()`, optimisers and
DDP-style hooks see ordinary `.grad` tensors.

Every tensor here is a torch CUDA tensor used as a memory handle; all arithmetic is in libpt_b200.so.
"""
from __future__ import annotations

import os
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import ops
from .ops import BF16, F32, OUT_BF16, OUT_F32, OUT_F32_ATOMIC_ADD



class Var:
    """An activation on the tape: `data` (bf16 [.., C] unless noted) and its gradient slot."""
    __slots__ = ("data", "grad", "owned", "needs_grad")

    def __init__(self, data: torch.Tensor, needs_grad: bool = True):
        self.data = data
        self.grad: Optional[torch.Tensor] = None
        self.owned = False
        self.needs_grad = needs_grad


class SideLane:
    """A second stream for backward work that nothing downstream waits for (bias gradients: only the optimiser / the gradient
    exchange read them).  A 128-thread column-sum CTA fits beside a persistent GEMM or attention CTA on the same SM, so on its own
    stream it runs in the resources and kernel-boundary gaps the main stream leaves idle (in-graph: parallel branches) instead of
    taking a slot in the serial kernel sequence (183 launches, 1.17 ms of a 43 ms step).  Tensors read on the lane are kept alive until
    the join."""

    def __init__(self, device):
        self.stream = torch.cuda.Stream(device)
        self.keep: List[torch.Tensor] = []
        self.dirty = False

    def run(self, fn: Callable[[], None], keep: Sequence[torch.Tensor] = ()) -> None:
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            fn()
        self.keep.extend(keep)
        self.dirty = True

    def join(self) -> None:
        if self.dirty:
            torch.cuda.current_stream().wait_stream(self.stream)
            self.dirty = False
            self.keep.clear()


# Off by default: a same-box A/B of the bench step (two runs each, 20 graph replays) gave 44.32 ms without and 44.40 ms with the lane --
# the column sums do overlap, but a persistent GEMM whose CTAs find an SM still busy with them starts that SM late, and the two
# effects cancel.  Kept behind PT_SIDE_LANE=1 for runs where the bias gradients are a larger share.
SIDE_LANE = os.environ.get("PT_SIDE_LANE", "0") == "1"


class PackCache:
    """bf16 GEMM-layout copies of fp32 parameters.

    Two kinds of entries:
      * static  -- views into an optimiser-owned bf16 shadow of the flat master buffer (`optim.FusedClipAdamW`): the AdamW kernel
        writes them, nothing is ever re-packed.  Guarded by the parameters' version counters, so an in-place write from outside
        (`load_state_dict`, `p.data.copy_`) refreshes the slice before it is used.
      * cached  -- packed on demand and re-packed when a parameter's version counter / storage moves (any torch optimiser).  While
        the current stream is being CAPTURED the re-pack always runs, into the same buffer: a captured step must contain the
        re-pack kernels, or its GEMMs would read the weights frozen at capture time while the optimiser updates the fp32 masters
        between replays.
    """

    def __init__(self):
        self._d: Dict[tuple, Tuple[tuple, torch.Tensor]] = {}
        self.static: Dict[tuple, list] = {}     # key -> [versions, view, refresh()]
        self.lane: Optional[SideLane] = None    # created on first use (lives as long as the model's cache)
        self.epoch = 0      # bumped by optimisers that update parameters through raw pointers without maintaining a static shadow

    def add_static(self, kind: str, params: Sequence[torch.Tensor], view: torch.Tensor, refresh: Optional[Callable[[], None]]) -> None:
        key = (kind,) + tuple(id(p) for p in params)
        self.static[key] = [tuple(p._version for p in params), view, refresh, list(params)]

    def get(self, params: Sequence[torch.Tensor], kind: str) -> torch.Tensor:
        key = (kind,) + tuple(id(p) for p in params)
        st = self.static.get(key)
        if st is not None:
            ver = tuple(p._version for p in params)
            if ver != st[0]:
                if st[2] is not None:
                    st[2]()
                st[0] = ver
            return st[1]
        ver = (self.epoch,) + tuple((p._version, p.data_ptr()) for p in params)
        hit = self._d.get(key)
        capturing = torch.cuda.is_current_stream_capturing() if params[0].is_cuda else False
        if hit is not None and hit[0] == ver and not capturing:
            return hit[1]
        prev = hit[1] if hit is not None else None
        if kind == "conv":      # [Co, Ci, k] -> [Co, k*Ci]
            (w,) = params
            if not w.is_contiguous():
                raise ops._lib.PtError("conv weight is a non-contiguous view (optimiser-managed) but has no static bf16 shadow")
            out = ops.pack_conv_weight(w.detach(), out=prev)
        elif kind == "bias":    # fp32 concatenation of 1-D parameters (a single one is used in place)
            if len(params) == 1:
                out = params[0].detach()
            else:
                out = torch.cat([p.detach() for p in params], out=prev) if prev is not None else torch.cat([p.detach() for p in params])
        else:                   # "lin": rows of all params stacked, cast to bf16 ([N, K]; 1x1 convs are [N, K, 1])
            rows = sum(p.shape[0] for p in params)
            K = params[0].numel() // params[0].shape[0]
            out = prev if prev is not None else torch.empty(rows, K, dtype=BF16, device=params[0].device)
            r = 0
            for p in params:
                ops.cast_bf16(p.detach().reshape(p.shape[0], K), out[r:r + p.shape[0]])
                r += p.shape[0]
        self._d[key] = (ver, out)
        return out


class Tape:
    def __init__(self, cache: PackCache, recording: bool = True):
        self.cache = cache
        self.recording = recording
        self.bwd: List[Callable[[], None]] = []
        self.pgrads: Dict[int, torch.Tensor] = {}
        self.params: Dict[int, torch.Tensor] = {}
        self.post: List[Callable[[], None]] = []   # run after the reverse sweep
        self.pgrad_order: List[Tuple[Sequence[torch.Tensor], torch.Tensor, str]] = []   # (params, buffer, kind) in completion order
        self.grad_alloc: Optional[Callable[[Sequence[torch.Tensor], str], Optional[torch.Tensor]]] = None   # flat-buffer provider (dp.GradSync)
        self.on_ready: Optional[Callable[[List[Tuple[Sequence[torch.Tensor], torch.Tensor, str]]], None]] = None
        # inference only: step-invariant cross-attention K/V projections of the text encoding, keyed by attention module
        # (the sampler passes the same dict to each of its 100 denoiser forwards)
        self.kv_cache: Optional[Dict[int, "Var"]] = None
        # cross-attention K/V of all layers as ONE projection of the text encoding: id(attention module) -> (Var, k_off, v_off)
        self.kv_group: Dict[int, Tuple["Var", int, int]] = {}
        # inference only (classifier-free guidance): rows [0, cond_rows) of the batch are conditioned on the context, the rows after
        # them have the null (all-zero) context, whose cross-attention update is the to_out bias alone (BasicTransformerBlock._fwd)
        self.cond_rows: Optional[int] = None

    def record(self, fn: Callable[[], None]) -> None:
        if self.recording:
            self.bwd.append(fn)

    # ---- parameter-gradient buffers.  One buffer per GROUP of parameters (a single one, or the stacked rows of a fused QKV / KV /
    # time-projection weight), fp32, accumulated into by the backward kernels.  Kinds:
    #   "plain"  the buffer has the parameter's own layout
    #   "cat"    [sum rows, K]: row slices are the gradients of the group's parameters
    #   "conv"   k=3 conv weight [Co, Ci, 3] accumulated TAP-MAJOR as [Co, 3, Ci] (the GEMM layout: contiguous output columns, so the
    #            stream-K flush uses vector REDs, and the flat master / shadow of the fused optimiser need no permutation); the
    #            gradient handed to torch is the permuted VIEW [Co, Ci, 3] of it.
    def _register(self, params: Sequence[torch.Tensor], kind: str, buf: torch.Tensor) -> None:
        if kind == "plain":
            (p,) = params
            self.pgrads[id(p)] = buf.view(p.shape)
            self.params[id(p)] = p
        elif kind == "conv":
            (p,) = params
            Co, Ci, k = p.shape
            packed = buf.view(Co, k, Ci)
            g = packed.permute(0, 2, 1)
            g._pt_buf = packed  # type: ignore[attr-defined]
            self.pgrads[id(p)] = g
            self.params[id(p)] = p
        else:
            rows = sum(p.shape[0] for p in params)
            K = params[0].numel() // params[0].shape[0]
            cat = buf.view(rows, K)
            r = 0
            for p in params:
                v = cat[r:r + p.shape[0]].view(p.shape)
                v._pt_buf = cat  # type: ignore[attr-defined]
                self.pgrads[id(p)] = v
                self.params[id(p)] = p
                r += p.shape[0]

    def _grad_buf(self, params: Sequence[torch.Tensor], kind: str) -> torch.Tensor:
        g = self.pgrads.get(id(params[0]))
        if g is None:
            n = sum(p.numel() for p in params)
            buf = self.grad_alloc(params, kind) if self.grad_alloc is not None else None
            if buf is None:
                buf = torch.zeros(n, dtype=F32, device=params[0].device)
            self._register(params, kind, buf)
            self.pgrad_order.append((list(params), buf, kind))
            g = self.pgrads[id(params[0])]
        return getattr(g, "_pt_buf", g)

    def rebind(self, params: Sequence[torch.Tensor], kind: str, buf: torch.Tensor) -> None:
        """Point the gradients of `params` at `buf` (dp.GradSync moves the first step's buffers into its flat buffer)."""
        self._register(params, kind, buf)

    def pgrad(self, p: torch.Tensor) -> torch.Tensor:
        return self._grad_buf([p], "plain")

    def pgrad_cat(self, params: Sequence[torch.Tensor]) -> torch.Tensor:
        """One fp32 buffer [sum rows, K] whose row slices are the gradients of `params` (fused QKV / KV weights)."""
        return self._grad_buf(params, "cat")

    def pgrad_conv(self, p: torch.Tensor) -> torch.Tensor:
        """fp32 [Co, 3, Ci] tap-major accumulation buffer of a k=3 conv weight (its torch gradient is the permuted view)."""
        return self._grad_buf([p], "conv")

    def side_colsum(self, x2d: torch.Tensor, out: torch.Tensor) -> None:
        """out[c] += sum_r x2d[r, c] (a bias gradient), off the critical path when a side lane is enabled."""
        if not SIDE_LANE or not x2d.is_cuda:
            ops.colsum(x2d, out)
            return
        if self.cache.lane is None:
            self.cache.lane = SideLane(x2d.device)
        self.cache.lane.run(lambda: ops.colsum(x2d, out, lite=True), keep=(x2d, out))

    def join_side(self) -> None:
        if self.cache.lane is not None:
            self.cache.lane.join()

    def backward(self) -> None:
        done = 0
        for fn in reversed(self.bwd):
            fn()
            if self.on_ready is not None and len(self.pgrad_order) > done:
                # every parameter feeds exactly one op, so its gradient is final when that op's backward returns
                self.on_ready(self.pgrad_order[done:])
                done = len(self.pgrad_order)
        self.bwd = []
        self.join_side()
        for fn in self.post:
            fn()
        self.post = []


def accum(v: Var, g: torch.Tensor, owned: bool = True) -> None:
    """Accumulate gradient `g` into `v` (g must be contiguous, same shape as v.data)."""
    if not v.needs_grad:
        return
    if v.grad is None:
        v.grad, v.owned = g, owned
    elif v.owned:
        ops.add_(v.grad, g, out=v.grad)
    else:
        v.grad = ops.add_(v.grad, g)
        v.owned = True


def _wgrad_gemm(dy2d_op, x2d_op, seg, N: int, K: int, out: torch.Tensor, out_stride_m: int) -> None:
    """dW[N, K] += dy^T x: fp32 atomic-accumulate output, scheduled stream-K by the library (the few-tile / long-K weight
    gradients load every SM evenly whatever the tile count)."""
    ops.gemm([dy2d_op], [x2d_op], [seg], N, K, out, out_strides=(out_stride_m, 0, 0), out_mode=OUT_F32_ATOMIC_ADD)


# ------------------------------------------------------------------------------------------------ linear / 1x1 conv
def linear(tape: Tape, x: Var, wparams: Sequence[torch.Tensor], bias: Optional[Sequence[torch.Tensor]] = None,
           residual: Optional[Var] = None, out_f32: bool = False, out: Optional[torch.Tensor] = None) -> Var:
    """y[M, N] = x[M, K] @ W^T (+ bias) (+ residual).  `wparams`: one or more fp32 parameters whose rows are stacked
    (nn.Linear [N, K] or 1x1 nn.Conv1d [N, K, 1]).  out: a contiguous tensor of y's shape and dtype to write into (a row range of
    a larger activation) instead of a new one."""
    xd = x.data
    K = xd.shape[-1]
    x2 = xd.reshape(-1, K)
    M = x2.shape[0]
    wp = tape.cache.get(wparams, "lin")
    N = wp.shape[0]
    shape = xd.shape[:-1] + (N,)
    if out is None:
        out = torch.empty(shape, dtype=F32 if out_f32 else BF16, device=xd.device)
    elif out.shape != shape or out.dtype != (F32 if out_f32 else BF16) or not out.is_contiguous():
        raise ops._lib.PtError(f"linear: out must be a contiguous {tuple(shape)} tensor, got {tuple(out.shape)} {out.dtype}")
    res = residual.data.reshape(M, N) if residual is not None else None
    ops.gemm([ops.operand(x2, True)], [ops.operand(wp, True)], [ops.segment(K)], M, N, out,
             out_mode=OUT_F32 if out_f32 else OUT_BF16, bias=tape.cache.get(bias, "bias") if bias is not None else None, residual=res)
    y = Var(out)

    def bwd():
        dy = y.grad
        if dy is None:
            return
        if out_f32:
            dy = ops.cast_bf16(dy)
        dy2 = dy.reshape(M, N)
        if bias is not None:
            tape.side_colsum(dy2, tape.pgrad_cat(bias) if len(bias) > 1 else tape.pgrad(bias[0]))
        gw = (tape.pgrad_cat(wparams) if len(wparams) > 1 else tape.pgrad(wparams[0])).view(N, K)
        _wgrad_gemm(ops.operand(dy2, False), ops.operand(x2, False), ops.segment(M), N, K, gw, K)
        if x.needs_grad:
            dx = torch.empty_like(x2) if (x.grad is None or not x.owned) else x.grad.reshape(M, K)
            prev = x.grad.reshape(M, K) if x.grad is not None else None
            ops.gemm([ops.operand(dy2, True)], [ops.operand(wp, False)], [ops.segment(N)], M, K, dx, residual=prev)
            x.grad, x.owned = dx.view(xd.shape), True
        if residual is not None:
            accum(residual, dy.view(residual.data.shape) if not out_f32 else dy.view(residual.data.shape), owned=False)

    tape.record(bwd)
    return y


# ------------------------------------------------------------------------------------------------ conv k=3
class TimeShift:
    """Per-(batch, channel) additive shift for conv1 of a resnet: a column slice of the batched time projection
    `proj` fp32 [B, total]; `dproj` collects its gradient."""

    def __init__(self, proj: torch.Tensor, dproj: Optional[torch.Tensor], offset: int):
        self.proj, self.dproj, self.offset = proj, dproj, offset


CONV_SWAP = os.environ.get("PT_CONV_NO_SWAP") is None


def _swap_tile(L: int, rows: int) -> int:
    """Tile width for running a k=3 convolution with the WEIGHTS on the 128-row side of the tile (M = channels, N = L, transposed
    output), or 0 to keep the rows of x there.  With at most 96 rows per sample (94 at level 3 of the bench model) a 128-row tile per
    sample is 27 % zero padding; the channel count is a multiple of 128 and the tile width can be L rounded up to 64 / 96.
    Measured (tools/conv_streamk_probe.py, B = 32): 49.3 vs 52.6 us at 94 x 1280 -> 1280, 90.6 vs 92.3 at 2560 -> 1280; at 188 rows
    (tile width 192 vs two row tiles) the two forms tie, so those keep the rows of x on the rows; the step gains 0.25 ms."""
    if not CONV_SWAP or rows % 128 != 0 or L > 96:
        return 0
    bn = 64 if L <= 64 else 96
    return bn if L / bn > L / 128 + 0.08 else 0


def conv3(tape: Tape, x: Var, wparam: torch.Tensor, bias: torch.Tensor, stride: int = 1,
          tshift: Optional[TimeShift] = None, residual: Optional[Var] = None) -> Var:
    """Conv1d(k=3, padding=1, stride 1|2) on channels-last x[B, L, Ci] as an implicit GEMM: three K segments whose
    A tile is the input shifted by -1/0/+1 rows (TMA zero fill = padding).  Optional fused time shift and residual."""
    xd = x.data
    B, L, Ci = xd.shape
    wp = tape.cache.get([wparam], "conv")      # [Co, 3*Ci]
    Co = wp.shape[0]
    Lo = L if stride == 1 else (L - 1) // 2 + 1
    out = torch.empty(B, Lo, Co, dtype=BF16, device=xd.device)
    if stride == 1:
        a_ops = [ops.operand(xd, True, batched=True)]
        taps = [(0, t - 1) for t in range(3)]                 # (A map, row shift)
    else:
        a_ops = [ops.operand(xd[:, 0::2], True, batched=True), ops.operand(xd[:, 1::2], True, batched=True)]
        taps = [(1, -1), (0, 0), (1, 0)]                      # in row 2l-1 = odd[l-1], 2l = even[l], 2l+1 = odd[l]
    segs = [ops.segment(Ci, a_idx=ai, a_shift=sh, b_k0=t * Ci) for t, (ai, sh) in enumerate(taps)]
    bz2 = tshift.proj[:, tshift.offset:] if tshift is not None else None
    sw = _swap_tile(L, Co) if stride == 1 else 0
    if sw:
        # weights on the rows: out^T[co, l] = sum_t W[co, t*Ci : (t+1)*Ci] . x[l + t - 1, :]
        segs_w = [ops.segment(Ci, a_k0=t * Ci, b_shift=t - 1) for t in range(3)]
        ops.gemm([ops.operand(wp, True)], a_ops, segs_w, Co, Lo, out, out_strides=(Co, Lo * Co, 0), nz2=B,
                 bias=bias.detach(), bias_z2=bz2, bias_z2_stride=tshift.proj.stride(0) if tshift is not None else 0,
                 residual=residual.data if residual is not None else None, res_strides=(Co, Lo * Co, 0), block_n=sw, out_transposed=True)
    else:
        ops.gemm(a_ops, [ops.operand(wp, True)], segs, Lo, Co, out, out_strides=(Co, Lo * Co, 0), nz2=B,
                 bias=bias.detach(), bias_z2=bz2, bias_z2_stride=tshift.proj.stride(0) if tshift is not None else 0,
                 residual=residual.data if residual is not None else None, res_strides=(Co, Lo * Co, 0))
    y = Var(out)

    def bwd():
        dy = y.grad
        if dy is None:
            return
        tape.side_colsum(dy.view(B * Lo, Co), tape.pgrad(bias))
        if tshift is not None and tshift.dproj is not None:
            ops.batch_colsum(dy, tshift.dproj[:, tshift.offset:], tshift.dproj.stride(0))
        # weight gradient: MN-major x MN-major GEMMs accumulated (fp32 atomics, stream-K) into the tap-major [Co, 3, Ci] buffer
        g3 = tape.pgrad_conv(wparam)
        dy_op = ops.operand(dy, False, batched=True)
        if stride == 1:
            # the three taps in ONE stream-K launch: z2 = tap shifts the rows of x by tap - 1 and the output by tap * Ci
            seg = ops.segment(Lo, b_k0=-1, b_k0_z2=1, nrep=B, rep_is_batch=True)
            ops.gemm([dy_op], [ops.operand(xd, False, batched=True)], [seg], Co, Ci, g3, out_strides=(3 * Ci, Ci, 0), nz2=3,
                     out_mode=OUT_F32_ATOMIC_ADD)
        else:
            for t, (ai, sh) in enumerate(taps):
                xs = xd[:, 0::2] if ai == 0 else xd[:, 1::2]
                seg = ops.segment(Lo, b_k0=sh, nrep=B, rep_is_batch=True)
                ops.gemm([dy_op], [ops.operand(xs, False, batched=True)], [seg], Co, Ci, g3[:, t],
                         out_strides=(3 * Ci, 0, 0), out_mode=OUT_F32_ATOMIC_ADD)
        if x.needs_grad:
            dy_k = ops.operand(dy, True, batched=True)
            wp_mn = ops.operand(wp, False)
            if stride == 1:
                own = x.grad is not None and x.owned
                dx = x.grad if own else torch.empty_like(xd)
                swx = _swap_tile(L, Ci)
                if swx:
                    # dx^T[ci, l] = sum_t W[:, t*Ci + ci]^T . dy[l + 1 - t, :]: the weights (read transposed in place) on the rows
                    segs_dx = [ops.segment(Co, a_shift=t * Ci, b_shift=1 - t) for t in range(3)]
                    ops.gemm([wp_mn], [dy_k], segs_dx, Ci, L, dx, out_strides=(Ci, L * Ci, 0), nz2=B,
                             residual=x.grad, res_strides=(Ci, L * Ci, 0), block_n=swx, out_transposed=True)
                else:
                    segs_dx = [ops.segment(Co, a_shift=1 - t, b_shift=t * Ci) for t in range(3)]
                    ops.gemm([dy_k], [wp_mn], segs_dx, L, Ci, dx, out_strides=(Ci, L * Ci, 0), nz2=B,
                             residual=x.grad, res_strides=(Ci, L * Ci, 0))
                x.grad, x.owned = dx, True
            else:
                dx = torch.empty_like(xd)
                ev, od = dx[:, 0::2], dx[:, 1::2]
                # even input rows 2l' feed tap 1 of output l'; odd rows 2l'+1 feed tap 0 of output l'+1 and tap 2 of output l'
                ops.gemm([dy_k], [wp_mn], [ops.segment(Co, b_shift=Ci)], ev.shape[1], Ci, ev, out_strides=(2 * Ci, L * Ci, 0), nz2=B)
                if od.shape[1] > 0:
                    ops.gemm([dy_k], [wp_mn], [ops.segment(Co, a_shift=1, b_shift=0), ops.segment(Co, a_shift=0, b_shift=2 * Ci)],
                             od.shape[1], Ci, od, out_strides=(2 * Ci, L * Ci, 0), nz2=B)
                accum(x, dx, owned=True)
        if residual is not None:
            accum(residual, dy, owned=False)

    tape.record(bwd)
    return y


# ------------------------------------------------------------------------------------------------ norms
def groupnorm(tape: Tape, x: Var, gamma: torch.Tensor, beta: torch.Tensor, eps: float, act: bool, groups: int = 32) -> Var:
    yd, stats = ops.groupnorm_fwd(x.data, gamma.detach(), beta.detach(), groups, eps, act)
    y = Var(yd)

    def bwd():
        if y.grad is None:
            return
        if not x.needs_grad:
            ops.groupnorm_bwd(y.grad, x.data, stats, gamma.detach(), beta.detach(), tape.pgrad(gamma), tape.pgrad(beta), groups, act)
            return
        # the residual branch usually reached x first: fold that gradient into this pass instead of a separate add kernel
        prev = x.grad
        dx = ops.groupnorm_bwd(y.grad, x.data, stats, gamma.detach(), beta.detach(), tape.pgrad(gamma), tape.pgrad(beta), groups, act,
                               dx_add=prev, out=prev if (prev is not None and x.owned) else None)
        x.grad, x.owned = dx, True

    tape.record(bwd)
    return y


def layernorm(tape: Tape, x: Var, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> Var:
    xd = x.data
    Cc = xd.shape[-1]
    x2 = xd.reshape(-1, Cc)
    yd, rs = ops.layernorm_fwd(x2, gamma.detach(), beta.detach(), eps)
    y = Var(yd.view(xd.shape))

    def bwd():
        if y.grad is None:
            return
        prev = x.grad.reshape(-1, Cc) if x.grad is not None else None
        dx = ops.layernorm_bwd(y.grad.reshape(-1, Cc), x2, rs, gamma.detach(), tape.pgrad(gamma), tape.pgrad(beta), dx_add=prev)
        if x.needs_grad:
            x.grad, x.owned = dx.view(xd.shape), True

    tape.record(bwd)
    return y


# ------------------------------------------------------------------------------------------------ attention core
def attention_core(tape: Tape, q_src: Var, q_off: int, kv_src: Var, k_off: int, v_off: int, heads: int, C: int,
                   shared_kv: bool = False) -> Var:
    """softmax(Q K^T / sqrt(d)) V with Q = q_src[..., q_off:q_off+C], K/V column slices of kv_src (no mask, no dropout:
    diffusers AttnProcessor2_0 as the reference uses it).  q_src [B, Lq, Wq], kv_src [B, Lk, Wkv].  One fused tcgen05
    kernel forward (logits stay in TMEM), three backward (delta, dQ, dK/dV) that recompute the logits from the saved
    log-sum-exp; gradients land in place in column slices of fused-projection-shaped buffers.
    shared_kv: kv_src holds the K/V projections of SEVERAL attention layers side by side (one grouped GEMM over the text encoding);
    every layer owns its own columns, so its dK/dV are written straight into those columns of one shared gradient buffer."""
    qd, kvd = q_src.data, kv_src.data
    B, Lq, _ = qd.shape
    d = C // heads
    scale = d ** -0.5
    qv, kv_, vv = qd[:, :, q_off:q_off + C], kvd[:, :, k_off:k_off + C], kvd[:, :, v_off:v_off + C]
    o = torch.empty(B, Lq, C, dtype=BF16, device=qd.device)
    lse = torch.empty(B, heads, Lq, dtype=F32, device=qd.device)
    ops.attn_fwd(qv, kv_, vv, o, lse, heads, d, scale)
    y = Var(o)

    def bwd():
        do = y.grad
        if do is None:
            return
        same = q_src is kv_src
        dq_buf = torch.empty_like(qd)
        if shared_kv:
            if kv_src.grad is None:       # first of the group to run backward; every column is written by exactly one layer
                kv_src.grad, kv_src.owned = torch.empty_like(kvd), True
            dkv_buf = kv_src.grad
        else:
            dkv_buf = dq_buf if same else torch.empty_like(kvd)
        ops.attn_bwd(qv, kv_, vv, o, lse, do, dq_buf[:, :, q_off:q_off + C], dkv_buf[:, :, k_off:k_off + C],
                     dkv_buf[:, :, v_off:v_off + C], heads, d, scale)
        accum(q_src, dq_buf, owned=True)
        if not same and not shared_kv:
            accum(kv_src, dkv_buf, owned=True)

    tape.record(bwd)
    return y


# ------------------------------------------------------------------------------------------------ condition dropout
def cond_keep_mask(keep, B: int, device, who: str) -> torch.Tensor:
    """Validate a classifier-free-guidance keep mask -- bool / uint8 [B] on the batch's CUDA device, nonzero = keep the text --
    and return its uint8 view (no copy for a contiguous mask: a captured step reads the caller's buffer at every replay)."""
    if not torch.is_tensor(keep) or keep.dtype not in (torch.bool, torch.uint8) or tuple(keep.shape) != (B,) \
            or not keep.is_cuda or keep.device != torch.device(device):
        desc = f"{keep.dtype} {tuple(keep.shape)} on {keep.device}" if torch.is_tensor(keep) else type(keep).__name__
        raise ops._lib.PtError(f"{who}: cond_keep must be a bool or uint8 tensor [B] = [{B}] on {device}, got {desc}")
    keep = keep.contiguous()
    return keep.view(torch.uint8) if keep.dtype == torch.bool else keep


def cond_select(tape: Tape, enc: Var, keep: torch.Tensor) -> Var:
    """Condition dropout on a text encoding [B, L, D]: rows b with keep[b] == 0 become the null (all-zero) context.  The backward
    applies the same selection to the gradient, so a dropped sample sends nothing back to the text encoder."""
    ed = enc.data
    B = ed.shape[0]
    per = ed[0].numel()
    y = Var(torch.empty_like(ed))
    ops.call("cond_select_bf16", ops._p(ed), ops._p(keep), ops._p(y.data), B, per, ops._stream())

    def bwd():
        if y.grad is None:
            return
        g = y.grad if y.owned else torch.empty_like(y.grad)
        ops.call("cond_select_bf16", ops._p(y.grad), ops._p(keep), ops._p(g), B, per, ops._stream())
        accum(enc, g, owned=True)

    tape.record(bwd)
    return y


# ------------------------------------------------------------------------------------------------ small ops
def geglu(tape: Tape, u: Var) -> Var:
    ud = u.data
    u2 = ud.reshape(-1, ud.shape[-1])
    y = Var(ops.geglu_fwd(u2).view(ud.shape[:-1] + (ud.shape[-1] // 2,)))

    def bwd():
        if y.grad is None:
            return
        accum(u, ops.geglu_bwd(y.grad.reshape(-1, ud.shape[-1] // 2), u2).view(ud.shape), owned=True)

    tape.record(bwd)
    return y


def add(tape: Tape, a: Var, b: Var) -> Var:
    y = Var(ops.add_(a.data, b.data))

    def bwd():
        if y.grad is None:
            return
        accum(a, y.grad, owned=False)
        accum(b, y.grad, owned=False)

    tape.record(bwd)
    return y


def concat_channels(tape: Tape, a: Var, b: Var) -> Var:
    """torch.cat([a, b], dim=channel) on channels-last tensors (unet_blocks.py:184,497)."""
    B, L, Ca = a.data.shape
    Cb = b.data.shape[2]
    out = torch.empty(B, L, Ca + Cb, dtype=BF16, device=a.data.device)
    ops.copy2d(a.data, Ca, out, Ca + Cb, B * L, Ca)
    ops.copy2d(b.data, Cb, out[:, :, Ca:], Ca + Cb, B * L, Cb)
    y = Var(out)

    def bwd():
        if y.grad is None:
            return
        g = y.grad
        ga = torch.empty_like(a.data)
        gb = torch.empty_like(b.data)
        ops.copy2d(g, Ca + Cb, ga, Ca, B * L, Ca)
        ops.copy2d(g[:, :, Ca:], Ca + Cb, gb, Cb, B * L, Cb)
        accum(a, ga, owned=True)
        accum(b, gb, owned=True)

    tape.record(bwd)
    return y


def upsample2(tape: Tape, x: Var) -> Var:
    y = Var(ops.upsample2_fwd(x.data))

    def bwd():
        if y.grad is None:
            return
        accum(x, ops.upsample2_bwd(y.grad), owned=True)

    tape.record(bwd)
    return y


def silu_f32(tape: Tape, x: Var) -> Var:
    """bf16(silu(x)) of a small fp32 tensor (time embedding path: resnet.py:255-257, TimestepEmbedding.act)."""
    y = Var(ops.silu_to_bf16(x.data))

    def bwd():
        if y.grad is None or not x.needs_grad:
            return
        g = ops.silu_bwd(x.data, ops.cast_f32(y.grad))
        if x.grad is None:
            x.grad, x.owned = g, True
        else:
            x.grad = x.grad + g   # fp32 [B, temb]: never hit on the reference path (single consumer)

    tape.record(bwd)
    return y


# ------------------------------------------------------------------------------------------------ autograd bridge
class TapeFunction(torch.autograd.Function):
    """Runs `runner(tape, *tensor_inputs)` -> (outputs, finish) once; `finish(tape, grad_outputs)` seeds the output
    gradients, after which the tape is swept in reverse and parameter / input gradients are handed to autograd."""

    @staticmethod
    def forward(ctx, runner, cache, n_in, *args):
        ins, params = args[:n_in], args[n_in:]
        need = any(ctx.needs_input_grad[3:])
        tape = Tape(cache, recording=need)
        outs, seed, in_grads = runner(tape, *ins)
        ctx.tape, ctx.seed, ctx.in_grads, ctx.n_in, ctx.params = tape, seed, in_grads, n_in, params
        ctx.mark_non_differentiable(*[o for o in outs if not o.is_floating_point()])
        return outs if len(outs) > 1 else outs[0]

    @staticmethod
    def backward(ctx, *gouts):
        tape = ctx.tape
        ctx.seed([g.contiguous() if g is not None else None for g in gouts])
        tape.backward()
        gin = ctx.in_grads()
        gparams = tuple(tape.pgrads.get(id(p)) if ctx.needs_input_grad[3 + ctx.n_in + i] else None for i, p in enumerate(ctx.params))
        ctx.tape = None
        return (None, None, None) + tuple(gin) + gparams


def get_cache(module) -> PackCache:
    c = module.__dict__.get("_pt_pack_cache")
    if c is None:
        c = PackCache()
        module.__dict__["_pt_pack_cache"] = c
    return c


def run_module(module, body, inputs, kinds, out_kind="ncl", multi=False):
    """Public-forward helper: convert reference-layout inputs to tape Vars, run `body(tape, *vars)`, convert the
    result back and bridge to autograd.  kinds: 'ncl' fp32 [B, C, L] activation, 'blc' float [B, L, C] activation,
    'f32' small fp32 tensor kept as is (differentiable), 'raw' passed through (no gradient).
    multi: `body` returns a list of Vars (the down blocks return the hidden state AND the skip states); the same Var may
    appear more than once (the reference returns the last skip state as the hidden state too) -- its gradients add up."""
    params = [p for p in module.parameters()]
    cache = get_cache(module)
    for t in inputs:
        if not t.is_cuda:
            raise ops._lib.PtError(f"{type(module).__name__}: inputs must be CUDA tensors; there is no CPU fallback")

    def runner(tape, *ins):
        vs = []
        for t, k in zip(ins, kinds):
            if k == "ncl":
                vs.append(Var(ops.ncl_to_nlc(t.detach().float().contiguous())))
            elif k == "blc":
                vs.append(Var(ops.cast_bf16(t.detach().float().contiguous())))
            elif k == "f32":
                vs.append(Var(t.detach().float().contiguous()))
            else:
                vs.append(t.detach())
        res = body(tape, *vs)
        yvs = list(res) if multi else [res]
        outs = tuple(ops.nlc_to_ncl(v.data) if out_kind == "ncl" else ops.cast_f32(v.data) for v in yvs)

        def seed(gouts):
            for v, g in zip(yvs, gouts):
                if g is None:
                    continue
                gg = ops.ncl_to_nlc(g.float().contiguous()) if out_kind == "ncl" else ops.cast_bf16(g.float().contiguous())
                accum(v, gg, owned=True)

        def in_grads():
            r = []
            for v, k in zip(vs, kinds):
                if k == "raw" or v.grad is None:
                    r.append(None)
                elif k == "ncl":
                    r.append(ops.nlc_to_ncl(v.grad))
                elif k == "blc":
                    r.append(ops.cast_f32(v.grad))
                else:
                    r.append(v.grad)
            return r

        return outs, seed, in_grads

    return TapeFunction.apply(runner, cache, len(inputs), *inputs, *params)
