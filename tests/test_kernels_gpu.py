"""GPU: each bandwidth-bound kernel against a plain torch fp32 statement of the same formula, and the RVQ kernels
bit-exactly against the C oracle and the committed golden vectors (through the C ABI)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from util import ROOT, rel

pytestmark = pytest.mark.gpu


def bf(x):
    return x.to(torch.bfloat16)


def gen(seed=0):
    return torch.Generator(device="cuda").manual_seed(seed)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("B,L,C,act", [(2, 50, 64, True), (3, 94, 320, True), (2, 188, 1920, False), (2, 33, 2560, True), (3, 752, 320, True),
                                       (2, 752, 640, True), (2, 5, 64, True)])
def test_groupnorm_fwd_bwd(cuda, B, L, C, act, fused):
    """fused: pt_groupnorm_fwd (the sample-resident cluster kernel where a sample fits; 752 x 640 fits forward but not backward; L = 5
    leaves three CTAs of a cluster without rows); else the streaming statistics + apply pair.  pt_groupnorm_bwd picks by itself."""
    from prompt_tts_b200 import ops
    g = gen(1)
    x = bf(torch.randn(B, L, C, device=cuda, generator=g) * 2 + 0.5)
    gamma = torch.randn(C, device=cuda, generator=g)
    beta = torch.randn(C, device=cuda, generator=g)
    dy = bf(torch.randn(B, L, C, device=cuda, generator=g))
    if fused:
        y, stats = ops.groupnorm_fwd(x, gamma, beta, 32, 1e-5, act)
        ref_stats = ops.groupnorm_stats(x, 32, 1e-5)
        assert rel(stats, ref_stats) < 1e-4
    else:
        stats = ops.groupnorm_stats(x, 32, 1e-5)
        y = ops.groupnorm_apply(x, stats, gamma, beta, 32, act)
    xr = x.float().transpose(1, 2).requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    yr = F.group_norm(xr, 32, gr, br, 1e-5)
    yr = F.silu(yr) if act else yr
    yr.backward(dy.float().transpose(1, 2))
    assert rel(y.float().transpose(1, 2), yr) < 6e-3
    dgam, dbet = torch.zeros(C, device=cuda), torch.zeros(C, device=cuda)
    dx = ops.groupnorm_bwd(dy, x, stats, gamma, beta, dgam, dbet, 32, act)
    assert rel(dx.float().transpose(1, 2), xr.grad) < 8e-3
    assert rel(dgam, gr.grad) < 2e-3 and rel(dbet, br.grad) < 2e-3
    # fused accumulation of a gradient that reached x through another branch, in place
    prev = bf(torch.randn(B, L, C, device=cuda, generator=g))
    acc = prev.clone()
    out = ops.groupnorm_bwd(dy, x, stats, gamma, beta, torch.zeros_like(dgam), torch.zeros_like(dbet), 32, act, dx_add=acc, out=acc)
    assert out.data_ptr() == acc.data_ptr()
    assert rel(acc.float().transpose(1, 2), xr.grad + prev.float().transpose(1, 2)) < 8e-3


@pytest.mark.parametrize("M,C", [(100, 64), (4099, 320), (777, 768), (513, 1280)])
def test_layernorm_fwd_bwd(cuda, M, C):
    from prompt_tts_b200 import ops
    g = gen(2)
    x = bf(torch.randn(M, C, device=cuda, generator=g) * 1.5 + 0.3)
    gamma, beta = torch.randn(C, device=cuda, generator=g), torch.randn(C, device=cuda, generator=g)
    dy, add = bf(torch.randn(M, C, device=cuda, generator=g)), bf(torch.randn(M, C, device=cuda, generator=g))
    y, rs = ops.layernorm_fwd(x, gamma, beta)
    xr = x.float().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    yr = F.layer_norm(xr, (C,), gr, br, 1e-5)
    yr.backward(dy.float())
    assert rel(y, yr) < 6e-3
    dgam, dbet = torch.zeros(C, device=cuda), torch.zeros(C, device=cuda)
    dx = ops.layernorm_bwd(dy, x, rs, gamma, dgam, dbet, dx_add=add)
    assert rel(dx, xr.grad + add.float()) < 8e-3
    assert rel(dgam, gr.grad) < 2e-3 and rel(dbet, br.grad) < 2e-3


@pytest.mark.parametrize("rows,n", [(37, 94), (1000, 550), (64, 752), (5, 1504), (9, 20)])
def test_softmax_fwd_bwd(cuda, rows, n):
    from prompt_tts_b200 import ops
    g = gen(3)
    ld = (n + 7) // 8 * 8
    S = torch.full((rows, ld), float("nan"), device=cuda)
    S[:, :n] = torch.randn(rows, n, device=cuda, generator=g) * 3
    P = torch.empty(rows, ld, device=cuda, dtype=torch.bfloat16)
    ops.softmax_fwd(S, P, rows, n, ld)
    ref = torch.softmax(S[:, :n], -1)
    assert rel(P[:, :n], ref) < 5e-3
    assert (P[:, n:(n + 3) // 4 * 4].float() == 0).all()      # the tail of the last 4-wide vector is written as zeros
    dP = torch.full((rows, ld), float("nan"), device=cuda)
    dP[:, :n] = torch.randn(rows, n, device=cuda, generator=g)
    dS = torch.empty(rows, ld, device=cuda, dtype=torch.bfloat16)
    ops.softmax_bwd(dP, P, dS, rows, n, ld, 0.25)
    Pf = P[:, :n].float()
    refd = 0.25 * Pf * (dP[:, :n] - (dP[:, :n] * Pf).sum(-1, keepdim=True))
    assert rel(dS[:, :n], refd) < 6e-3


# (B, H, Lq, Lk, d, fused): head dims of the tiny configs (8, 16), the text encoder (64) and the three UNet levels (40, 80, 160);
# ragged lengths (not multiples of the 64 / 128 tiles), cross attention with Lk != Lq, fused QKV / KV column-slice layouts
ATTN_CASES = [(2, 8, 24, 24, 8, True), (2, 8, 47, 33, 16, False), (1, 2, 128, 128, 40, True), (2, 3, 200, 150, 40, False),
              (2, 12, 131, 131, 64, True), (2, 8, 94, 550, 80, False), (2, 8, 188, 188, 160, True), (3, 8, 94, 129, 160, False)]


@pytest.mark.parametrize("B,H,Lq,Lk,d,fused", ATTN_CASES)
def test_fused_attention_fwd_bwd(cuda, B, H, Lq, Lk, d, fused):
    """pt_attn_fwd / pt_attn_bwd against the oracle's attention (oracle/ref_model.py:_attn, identity projections) in fp32."""
    import ref_model
    from prompt_tts_b200 import ops
    g = gen(11)
    C = H * d
    scale = d ** -0.5
    if fused:      # self attention on a fused [Q | K | V] projection, gradients written into a fused buffer
        qkv = bf(torch.randn(B, Lq, 3 * C, device=cuda, generator=g) * 1.5)
        q, k, v = qkv[:, :, :C], qkv[:, :, C:2 * C], qkv[:, :, 2 * C:]
        dbuf = torch.full_like(qkv, float("nan"))
        dq, dk, dv = dbuf[:, :, :C], dbuf[:, :, C:2 * C], dbuf[:, :, 2 * C:]
    else:          # cross attention: Q its own tensor, [K | V] fused
        q = bf(torch.randn(B, Lq, C, device=cuda, generator=g) * 1.5)
        kv = bf(torch.randn(B, Lk, 2 * C, device=cuda, generator=g) * 1.5)
        k, v = kv[:, :, :C], kv[:, :, C:]
        dq = torch.full_like(q, float("nan"))
        dkv = torch.full_like(kv, float("nan"))
        dk, dv = dkv[:, :, :C], dkv[:, :, C:]
    do = bf(torch.randn(B, Lq, C, device=cuda, generator=g))
    o = torch.full((B, Lq, C), float("nan"), device=cuda, dtype=torch.bfloat16)
    lse = torch.full((B, H, Lq), float("nan"), device=cuda)
    ops.attn_fwd(q, k, v, o, lse, H, d, scale)
    ops.attn_bwd(q, k, v, o, lse, do, dq, dk, dv, H, d, scale)
    torch.cuda.synchronize()

    # oracle: _attn with selector projections (to_q = I, to_k = [I 0], to_v = [0 I] on ctx = [k | v], to_out = I), so the
    # reference function computes exactly softmax(q k^T / sqrt d) v per head on our inputs
    eye, zero = torch.eye(C, device=cuda), torch.zeros(C, C, device=cuda)
    sd = {"a.to_q.weight": eye, "a.to_k.weight": torch.cat([eye, zero], 1), "a.to_v.weight": torch.cat([zero, eye], 1),
          "a.to_out.0.weight": eye, "a.to_out.0.bias": torch.zeros(C, device=cuda)}
    qf, kf, vf = (t.float().clone().requires_grad_(True) for t in (q, k, v))
    ref_o = ref_model._attn(sd, "a", qf, torch.cat([kf, vf], -1), H)
    sc = (qf.view(B, Lq, H, d).transpose(1, 2) @ kf.view(B, Lk, H, d).transpose(1, 2).transpose(-1, -2)) * scale
    ref_o.backward(do.float())
    assert rel(o, ref_o) < 4e-3, rel(o, ref_o)
    assert rel(lse, torch.logsumexp(sc, -1).detach()) < 1e-5
    assert rel(dq, qf.grad) < 8e-3 and rel(dk, kf.grad) < 8e-3 and rel(dv, vf.grad) < 8e-3, (rel(dq, qf.grad), rel(dk, kf.grad), rel(dv, vf.grad))
    # nothing outside the written slices was touched / nothing inside was left unwritten
    assert torch.isfinite(o.float()).all() and torch.isfinite(dq.float()).all() and torch.isfinite(dk.float()).all() and torch.isfinite(dv.float()).all()


@pytest.mark.parametrize("Lq,Lk,d", [(200, 330, 40), (130, 752, 64), (94, 550, 160)])
def test_fused_attention_rescale_path(cuda, Lq, Lk, d):
    """The forward is an online softmax that rescales a group's accumulator only when a row maximum grows by more than 2^8.  Random
    logits never do that, so force it: key norms ramp up along the sequence (every later 64-key tile raises the maximum by far more
    than the threshold, for both transform groups) and a few rows get the opposite sign (their maximum sits in the FIRST tile)."""
    from prompt_tts_b200 import ops
    g = gen(21)
    B, H = 2, 4
    C = H * d
    scale = d ** -0.5
    q = bf(torch.randn(B, Lq, C, device=cuda, generator=g))
    ramp = torch.linspace(0.05, 6.0, Lk, device=cuda)[None, :, None]
    kv = torch.randn(B, Lk, 2 * C, device=cuda, generator=g)
    kv[:, :, :C] = q[:, :1, :].float().sign() * kv[:, :, :C].abs() * ramp      # aligned with row 0 of q: logits grow with the key index
    kv = bf(kv)
    q = q.clone()
    q[:, 1::7] = -q[:, 1::7].abs() * q[:, :1, :].sign()                          # some rows see decreasing logits instead
    k, v = kv[:, :, :C], kv[:, :, C:]
    o = torch.full((B, Lq, C), float("nan"), device=cuda, dtype=torch.bfloat16)
    lse = torch.full((B, H, Lq), float("nan"), device=cuda)
    ops.attn_fwd(q, k, v, o, lse, H, d, scale)
    qh = q.float().view(B, Lq, H, d).transpose(1, 2)
    kh = k.float().view(B, Lk, H, d).transpose(1, 2)
    vh = v.float().view(B, Lk, H, d).transpose(1, 2)
    sc = (qh @ kh.transpose(-1, -2)) * scale
    spread = (sc.max(-1).values - sc[..., :64].max(-1).values).max().item()
    assert spread * 1.4427 > 8 * 3, f"the test must cross the rescale threshold several times (spread {spread})"
    ref = (torch.softmax(sc, -1) @ vh).transpose(1, 2).reshape(B, Lq, C)
    assert torch.isfinite(o.float()).all()
    assert rel(o, ref) < 4e-3, rel(o, ref)
    assert rel(lse, torch.logsumexp(sc, -1)) < 1e-5


def _attn_inputs(B, H, Lq, Lk, d, same, amp, seed=0):
    """bf16 inputs in the layouts the model uses (fused [Q|K|V] for self-attention, Q + fused [K|V] for cross-attention), every
    output prefilled with NaN so that an unwritten or corrupted element cannot hide."""
    g = gen(seed)
    C = H * d
    if same:
        qkv = bf(torch.randn(B, Lq, 3 * C, device="cuda", generator=g) * amp)
        q, k, v = qkv[:, :, :C], qkv[:, :, C:2 * C], qkv[:, :, 2 * C:]
        dbuf = torch.full_like(qkv, float("nan"))
        dq, dk, dv = dbuf[:, :, :C], dbuf[:, :, C:2 * C], dbuf[:, :, 2 * C:]
    else:
        q = bf(torch.randn(B, Lq, C, device="cuda", generator=g) * amp)
        kv = bf(torch.randn(B, Lk, 2 * C, device="cuda", generator=g) * amp)
        k, v = kv[:, :, :C], kv[:, :, C:]
        dq = torch.full_like(q, float("nan"))
        dkv = torch.full_like(kv, float("nan"))
        dk, dv = dkv[:, :, :C], dkv[:, :, C:]
    do = bf(torch.randn(B, Lq, C, device="cuda", generator=g))
    o = torch.full((B, Lq, C), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.full((B, H, Lq), float("nan"), device="cuda")
    return q, k, v, do, o, lse, dq, dk, dv


def _attn_oracle_errs(q, k, v, do, o, lse, dq, dk, dv, H, d, want_grads=True):
    """Squared-error sums against the oracle's attention (oracle/ref_model.py:_attn restated per head in fp32), one batch element
    at a time so the [H, Lq, Lk] fp32 matrices stay small at the bench shapes."""
    B, Lq, C = q.shape
    Lk = k.shape[1]
    scale = d ** -0.5
    num = {n: 0.0 for n in ("o", "lse", "dq", "dk", "dv")}
    den = dict(num)

    def heads(t, L):
        return t.float().reshape(L, H, d).transpose(0, 1)

    for b in range(B):
        qf, kf, vf = (heads(t[b], L).clone().requires_grad_(want_grads) for t, L in ((q, Lq), (k, Lk), (v, Lk)))
        s = (qf @ kf.transpose(-1, -2)) * scale
        of = torch.softmax(s, -1) @ vf
        pairs = [("o", heads(o[b], Lq), of.detach()), ("lse", lse[b], torch.logsumexp(s, -1).detach())]
        if want_grads:
            of.backward(heads(do[b], Lq))
            pairs += [("dq", heads(dq[b], Lq), qf.grad), ("dk", heads(dk[b], Lk), kf.grad), ("dv", heads(dv[b], Lk), vf.grad)]
        for n, a, r in pairs:
            num[n] += (a.float() - r).pow(2).sum().item()
            den[n] += r.pow(2).sum().item()
    return {n: (num[n] / (den[n] + 1e-30)) ** 0.5 for n in num if den[n] > 0}


# the seven attention shapes of one bench step (B = 32): three UNet levels self / cross, and the text encoder
FULL_ATTN = {"full_d40_self": (32, 8, 752, 752, 40, True), "full_d40_cross": (32, 8, 752, 550, 40, False),
             "full_d80_self": (32, 8, 376, 376, 80, True), "full_d80_cross": (32, 8, 376, 550, 80, False),
             "full_d160_self": (32, 8, 188, 188, 160, True), "full_d160_cross": (32, 8, 188, 550, 160, False),
             "full_text_d64": (32, 12, 550, 550, 64, True)}


@pytest.mark.parametrize("name", list(FULL_ATTN))
def test_fused_attention_bench_shapes_vs_oracle(cuda, name):
    """Every attention shape of the bench step against the fp32 oracle, inputs x1.5 (logit spread that makes some rows take the
    online-softmax rescale path), NaN-prefilled outputs.  Round 1's probe showed NaN in O at `full_d40_self` with exactly these inputs."""
    from prompt_tts_b200 import ops
    B, H, Lq, Lk, d, same = FULL_ATTN[name]
    q, k, v, do, o, lse, dq, dk, dv = _attn_inputs(B, H, Lq, Lk, d, same, 1.5)
    ops.attn_fwd(q, k, v, o, lse, H, d, d ** -0.5)
    ops.attn_bwd(q, k, v, o, lse, do, dq, dk, dv, H, d, d ** -0.5)
    torch.cuda.synchronize()
    for t in (o, lse, dq, dk, dv):
        assert torch.isfinite(t.float()).all()
    e = _attn_oracle_errs(q, k, v, do, o, lse, dq, dk, dv, H, d)
    assert e["o"] < 4e-3 and e["lse"] < 1e-5 and e["dq"] < 8e-3 and e["dk"] < 8e-3 and e["dv"] < 8e-3, e


@pytest.mark.parametrize("amp,iters", [(1.5, 200), (3.0, 40)])
def test_fused_attention_d40_self_repeat(cuda, amp, iters):
    """The round-1 failure was a race (one warp of a transform group lagging a tile behind the others while it rescales): run the
    level-0 self-attention forward many times on the same inputs and require finite, correct output EVERY time.  amp = 3 makes
    nearly every row rescale several times (it failed deterministically before the per-slot t_full barriers)."""
    from prompt_tts_b200 import ops
    B, H, Lq, Lk, d, same = FULL_ATTN["full_d40_self"]
    q, k, v, do, o, lse, dq, dk, dv = _attn_inputs(B, H, Lq, Lk, d, same, amp)
    ops.attn_fwd(q, k, v, o, lse, H, d, d ** -0.5)
    torch.cuda.synchronize()
    e = _attn_oracle_errs(q, k, v, do, o, lse, dq, dk, dv, H, d, want_grads=False)
    assert e["o"] < 4e-3 and e["lse"] < 1e-5, e
    o_ref, lse_ref = o.clone(), lse.clone()
    for it in range(iters):
        o.fill_(float("nan"))
        lse.fill_(float("nan"))
        ops.attn_fwd(q, k, v, o, lse, H, d, d ** -0.5)
        assert torch.isfinite(o.float()).all() and torch.isfinite(lse).all(), f"non-finite output at iteration {it}"
        # the kernel is deterministic for fixed inputs except for WHICH rows rescale when (nothing here depends on timing)
        assert rel(o, o_ref) < 4e-3 and rel(lse, lse_ref) < 1e-6, f"iteration {it}: {rel(o, o_ref)}"
    for it in range(max(2, iters // 20)):
        for t in (dq, dk, dv):
            t.fill_(float("nan"))
        ops.attn_bwd(q, k, v, o_ref, lse_ref, do, dq, dk, dv, H, d, d ** -0.5)
        assert all(torch.isfinite(t.float()).all() for t in (dq, dk, dv)), f"non-finite gradient at iteration {it}"


def test_fused_attention_properties_full_size(cuda):
    """Size-independent properties at the bench shape (32 x 8 heads x 752 x 752, d = 40), where a dense reference would
    need 2.3 GB per [B, H, Lq, Lk] matrix: rows of softmax sum to one (V = 1 -> O = 1), O is linear in V, and permuting the
    keys together with the values leaves O unchanged."""
    from prompt_tts_b200 import ops
    g = gen(12)
    B, H, L, d = 32, 8, 752, 40
    C = H * d
    qkv = bf(torch.randn(B, L, 3 * C, device=cuda, generator=g))
    q, k, v = qkv[:, :, :C], qkv[:, :, C:2 * C], qkv[:, :, 2 * C:]
    lse = torch.empty(B, H, L, device=cuda)

    def run(kk, vv):
        kv = torch.cat([kk, vv], -1)          # K and V must share one row stride (they are slices of one fused projection)
        o = torch.empty(B, L, C, device=cuda, dtype=torch.bfloat16)
        ops.attn_fwd(q, kv[:, :, :C], kv[:, :, C:], o, lse, H, d, d ** -0.5)
        return o.float()

    ones = torch.ones(B, L, C, device=cuda, dtype=torch.bfloat16)
    assert (run(k, ones) - 1).abs().max() < 8e-3
    o1 = run(k, v)
    o2 = run(k, bf(2 * v.float()))
    assert rel(o2, 2 * o1) < 4e-3
    perm = torch.randperm(L, device=cuda, generator=g)
    o3 = run(k[:, perm].contiguous(), v[:, perm].contiguous())
    assert rel(o3, o1) < 4e-3


def test_geglu_add_upsample_copy(cuda):
    from prompt_tts_b200 import ops
    g = gen(4)
    u = bf(torch.randn(300, 512, device=cuda, generator=g))
    dy = bf(torch.randn(300, 256, device=cuda, generator=g))
    y = ops.geglu_fwd(u)
    ur = u.float().requires_grad_(True)
    a, gt = ur.chunk(2, -1)
    yr = a * F.gelu(gt)
    yr.backward(dy.float())
    assert rel(y, yr) < 5e-3 and rel(ops.geglu_bwd(dy, u), ur.grad) < 6e-3
    for (Mg, Fg) in [(20011, 1280), (70, 8)]:   # more items than one grid sweep (two items per thread in flight) and a tiny one
        ub = bf(torch.randn(Mg, 2 * Fg, device=cuda, generator=g))
        dyb = bf(torch.randn(Mg, Fg, device=cuda, generator=g))
        ubr = ub.float().requires_grad_(True)
        ab, gb = ubr.chunk(2, -1)
        ybr = ab * F.gelu(gb)
        ybr.backward(dyb.float())
        assert rel(ops.geglu_fwd(ub), ybr) < 5e-3 and rel(ops.geglu_bwd(dyb, ub), ubr.grad) < 6e-3
    a2, b2 = bf(torch.randn(64, 320, device=cuda, generator=g)), bf(torch.randn(64, 320, device=cuda, generator=g))
    assert rel(ops.add_(a2, b2), a2.float() + b2.float()) < 5e-3
    x = bf(torch.randn(2, 47, 64, device=cuda, generator=g))
    up = ops.upsample2_fwd(x)
    assert torch.equal(up, x.repeat_interleave(2, dim=1))
    d = bf(torch.randn(2, 94, 64, device=cuda, generator=g))
    assert rel(ops.upsample2_bwd(d), d.float().view(2, 47, 2, 64).sum(2)) < 5e-3
    ncl = torch.randn(3, 70, 45, device=cuda, generator=g)
    nlc = ops.ncl_to_nlc(ncl)
    assert torch.equal(nlc, bf(ncl.transpose(1, 2)))
    assert torch.equal(ops.nlc_to_ncl(nlc), nlc.float().transpose(1, 2))
    w = torch.randn(96, 40, 3, device=cuda, generator=g)
    assert torch.equal(ops.pack_conv_weight(w), bf(w.permute(0, 2, 1).reshape(96, 120)))
    gp = torch.randn(96, 120, device=cuda, generator=g)
    gacc = torch.ones(96, 40, 3, device=cuda)
    ops.unpack_conv_wgrad(gp, gacc, accumulate=True)
    assert torch.allclose(gacc, 1 + gp.view(96, 3, 40).permute(0, 2, 1))
    xs = bf(torch.randn(5000, 10240, device=cuda, generator=g))
    cs = torch.zeros(10240, device=cuda)
    ops.colsum(xs, cs)
    assert rel(cs, xs.float().sum(0)) < 1e-4
    xb = bf(torch.randn(4, 300, 320, device=cuda, generator=g))
    bc = torch.full((4, 1000), 7.0, device=cuda)
    ops.batch_colsum(xb, bc[:, 100:], 1000)
    assert rel(bc[:, 100:420], xb.float().sum(1)) < 1e-4 and (bc[:, :100] == 7).all() and (bc[:, 420:] == 7).all()


def test_conv_in_out(cuda):
    from prompt_tts_b200 import ops
    from prompt_tts_b200.ops import _p, _stream, call
    g = gen(5)
    B, Cin, L, C = 3, 8, 75, 320
    x = torch.randn(B, Cin, L, device=cuda, generator=g)
    w = (torch.randn(C, Cin, 3, device=cuda, generator=g) * 0.2).requires_grad_(True)
    b = torch.randn(C, device=cuda, generator=g).requires_grad_(True)
    y = torch.empty(B, L, C, device=cuda, dtype=torch.bfloat16)
    call("conv_in_fwd", _p(x), _p(w.detach()), _p(b.detach()), _p(y), B, Cin, L, C, _stream())
    yr = F.conv1d(x, w, b, padding=1)
    assert rel(y.float().transpose(1, 2), yr) < 5e-3
    dy = bf(torch.randn(B, L, C, device=cuda, generator=g))
    yr.backward(dy.float().transpose(1, 2))
    dw, db = torch.zeros_like(w), torch.zeros_like(b)
    call("conv_in_bwd", _p(dy), _p(x), _p(dw), _p(db), B, Cin, L, C, _stream())
    assert rel(dw, w.grad) < 1e-4 and rel(db, b.grad) < 1e-4
    # conv_out
    h = bf(torch.randn(B, L, C, device=cuda, generator=g))
    wo = (torch.randn(8, C, 3, device=cuda, generator=g) * 0.1).requires_grad_(True)
    bo = torch.randn(8, device=cuda, generator=g).requires_grad_(True)
    yo = torch.empty(B, 8, L, device=cuda)
    call("conv_out_fwd", _p(h), _p(wo.detach()), _p(bo.detach()), _p(yo), B, C, L, 8, _stream())
    hr = h.float().transpose(1, 2).requires_grad_(True)
    yor = F.conv1d(hr, wo, bo, padding=1)
    assert rel(yo, yor) < 1e-5
    dyo = torch.randn(B, 8, L, device=cuda, generator=g)
    yor.backward(dyo)
    dh = torch.empty_like(h)
    dwo, dbo = torch.zeros_like(wo), torch.zeros_like(bo)
    call("conv_out_bwd", _p(dyo), _p(h), _p(wo.detach()), _p(dh), _p(dwo), _p(dbo), B, C, L, 8, _stream())
    assert rel(dh.float().transpose(1, 2), hr.grad) < 5e-3
    assert rel(dwo, wo.grad) < 1e-4 and rel(dbo, bo.grad) < 1e-4


def test_time_text_noise_mse(cuda):
    import ref_model
    from prompt_tts_b200 import ops
    from prompt_tts_b200.ops import _p, _stream, call
    from prompt_tts_b200.train import ddpm_tables
    t = torch.tensor([0, 1, 17, 500, 999], device=cuda)
    assert rel(ops.time_sinusoid(t, 320), ref_model.timestep_sinusoid(t, 320)) < 2e-5
    g = gen(6)
    x0, nz = torch.randn(5, 8, 40, device=cuda, generator=g), torch.randn(5, 8, 40, device=cuda, generator=g)
    sa, sb = ddpm_tables(device=cuda)
    xt = torch.empty_like(x0)
    call("add_noise", _p(x0), _p(nz), _p(t), _p(sa), _p(sb), _p(xt), 5, 320, _stream())
    assert rel(xt, ref_model.add_noise(x0, nz, t)) < 1e-6
    loss, dp = torch.zeros((), device=cuda), torch.empty_like(x0)
    call("mse_fwd_bwd", _p(xt), _p(nz), _p(loss), _p(dp), xt.numel(), 1.0, _stream())
    assert abs(loss.item() - F.mse_loss(xt, nz).item()) < 1e-5 and rel(dp, 2 * (xt - nz) / xt.numel()) < 1e-6
    ids = torch.randint(0, 150, (3, 24), device=cuda, generator=g).to(torch.int32)
    E_ = torch.randn(150, 64, device=cuda, generator=g)
    pe = ref_model.text_positional_encoding(24, 64, 24, cuda)
    y = torch.empty(3, 24, 64, device=cuda, dtype=torch.bfloat16)
    call("text_embed_fwd", _p(ids), _p(E_), _p(pe), _p(y), 3, 24, 64, 150, _stream())
    assert rel(y, F.embedding(ids.long(), E_) + pe[None]) < 4e-3


def _make_golden():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "oracle", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg


def _golden_rvq(name):
    mg = _make_golden()
    g = np.load(os.path.join(ROOT, "tests", "golden", f"rvq_{name}.npz"))
    seed, B, T, grid = int(g["seed"]), int(g["B"]), int(g["T"]), bool(g["grid"])
    return g, mg.rvq_codebooks(seed, grid), mg.rvq_latents(seed, B, T, grid)


@pytest.mark.parametrize("name", ["grid", "gauss"])
def test_rvq_matches_golden_and_oracle_bit_exact(cuda, name):
    import rvq_oracle
    from prompt_tts_b200 import ops
    g, cb, lat = _golden_rvq(name)
    codes = ops.rvq_encode(torch.from_numpy(lat).to(cuda), torch.from_numpy(cb).to(cuda)).cpu().numpy()
    assert np.array_equal(codes, rvq_oracle.encode(lat, cb))                  # bit-exact against the oracle
    if name == "grid":
        assert np.array_equal(codes, g["codes"].astype(np.int64))             # and against the encodec golden vectors
    else:
        assert (codes != g["codes"]).mean() < 1e-3
    dec = ops.rvq_decode(torch.from_numpy(g["codes"].astype(np.int64)).to(cuda), torch.from_numpy(cb).to(cuda)).cpu().numpy()
    assert np.array_equal(dec[:, :, : g["dec_slice"].shape[2]], g["dec_slice"])
    assert np.array_equal(dec, rvq_oracle.decode(g["codes"].astype(np.int64), cb))


def test_rvq_full_reference_batch_bit_exact(cuda):
    """One complete reference batch (32 clips x 900 frames, generate_code.py:29-34,94-96; Gaussian latents and codebooks):
    every one of the 230 400 codes equals the C oracle's, and against the encodec RVQ itself (transformers' line-for-line
    restatement, run on the host cores with its library GEMM; its codes and a hash of its decode are stored by
    oracle/make_golden.py) the only frames that may differ are fp64 near-ties, where the unspecified summation order of that GEMM
    decides (SURVEY 7.3-3d)."""
    import hashlib
    import rvq_oracle
    from prompt_tts_b200 import ops
    cb, lat = _make_golden().rvq_full_batch()
    g = np.load(os.path.join(ROOT, "tests", "golden", "rvq_full_batch.npz"))
    codes = ops.rvq_encode(torch.from_numpy(lat).to(cuda), torch.from_numpy(cb).to(cuda)).cpu().numpy()
    want = rvq_oracle.encode(lat, cb, threads=os.cpu_count() or 1)
    assert np.array_equal(codes, want), f"{(codes != want).sum()} of {codes.size} codes differ from the oracle"
    ref = g["codes"].astype(np.int64)
    assert ref.shape == codes.shape
    diff = codes != ref
    if diff.any():
        bad_frames = diff.any(axis=1)                          # [B, T]: a flip cascades to the later stages of the same frame
        sub = lat.transpose(0, 2, 1)[bad_frames].T[None]       # [1, 128, n_bad]
        _, margin = rvq_oracle.encode_fp64(np.ascontiguousarray(sub), cb)
        first = diff.transpose(0, 2, 1)[bad_frames].argmax(axis=1)            # first differing stage per bad frame
        m_first = margin[0].T[np.arange(len(first)), first]
        assert (m_first < 1e-4).all(), f"a clear (non-tie) decision differs from encodec: margins {m_first[:8]}"
    assert diff.mean() < 1e-3
    dec = ops.rvq_decode(torch.from_numpy(ref).to(cuda), torch.from_numpy(cb).to(cuda)).cpu().numpy()
    assert dec.dtype == np.float32 and dec.shape == (32, 128, 900)
    assert hashlib.sha256(np.ascontiguousarray(dec).tobytes()).hexdigest() == str(g["dec_sha256"])   # bit-equal to encodec's decode


def test_rvq_tensor_core_preselect_equals_exhaustive(cuda):
    """The two quantisers (tcgen05 pre-selection + exact re-rank, csrc/rvq_tc.cu; exhaustive fp32 search, csrc/rvq.cu) must give
    the same codes on everything: Gaussian data at several scales (the error bound scales with |r| |e|), grid-valued data with exact
    ties, zero frames, ragged frame counts -- and degenerate codebooks where hundreds of codes fall inside the rounding window, which
    must take the exhaustive fallback (duplicated codes: the FIRST index wins)."""
    import rvq_oracle
    from prompt_tts_b200 import ops
    g = gen(31)
    for scale_x, scale_e, B, T in [(1.0, 1.0, 5, 333), (30.0, 0.05, 2, 129), (1e-3, 4.0, 3, 64), (1.0, 1.0, 1, 1)]:
        cb = torch.randn(8, 1024, 128, device=cuda, generator=g) * scale_e
        lat = torch.randn(B, 128, T, device=cuda, generator=g) * scale_x
        lat[:, :, T // 2:T // 2 + 3] = 0.0
        a, b = ops.rvq_encode(lat, cb), ops.rvq_encode(lat, cb, exhaustive=True)
        assert torch.equal(a, b), (scale_x, scale_e, int((a != b).sum()))
    # fewer codebooks / smaller codebooks (K = 256), and values on a coarse grid (exact ties are common)
    cb = (torch.randint(-8, 9, (3, 256, 128), device=cuda, generator=g).float() / 16)
    lat = (torch.randint(-16, 17, (4, 128, 200), device=cuda, generator=g).float() / 16)
    a, b = ops.rvq_encode(lat, cb), ops.rvq_encode(lat, cb, exhaustive=True)
    assert torch.equal(a, b)
    assert np.array_equal(a.cpu().numpy(), rvq_oracle.encode(lat.cpu().numpy(), cb.cpu().numpy()))
    # degenerate: every code appears 8 times -> each maximum is an 8-way exact tie; and a codebook of 1024 near-identical codes
    base = torch.randn(8, 128, 128, device=cuda, generator=g)
    cb = base.repeat_interleave(8, dim=1).contiguous()
    lat = torch.randn(2, 128, 150, device=cuda, generator=g)
    a, b = ops.rvq_encode(lat, cb), ops.rvq_encode(lat, cb, exhaustive=True)
    assert torch.equal(a, b) and int((a % 8).max()) == 0
    cb = (torch.randn(1, 1, 128, device=cuda, generator=g) + 1e-4 * torch.randn(2, 1024, 128, device=cuda, generator=g)).contiguous()
    a, b = ops.rvq_encode(lat, cb), ops.rvq_encode(lat, cb, exhaustive=True)
    assert torch.equal(a, b)
    assert ops.rvq_encode.last_prepared.overflow_frames() > 0, "the near-identical codebook must have exercised the exhaustive fallback"
    # a prepared handle is reusable across calls and gives the same codes
    cb = torch.randn(8, 1024, 128, device=cuda, generator=g)
    prep = ops.rvq_prepare(cb)
    for _ in range(2):
        assert torch.equal(ops.rvq_encode(lat, cb, prepared=prep), ops.rvq_encode(lat, cb, exhaustive=True))


def test_rvq_ragged_and_properties(cuda):
    """LJSpeech-like batch (32 x 900 frames, reference layout generate_code.py:29-34): bit-exact against the oracle on a
    sample, plus size-independent properties: decode(encode(x)) reduces the residual at every stage; encode of an exact
    code vector sum returns codes whose decode reproduces the input."""
    import rvq_oracle
    from prompt_tts_b200 import ops
    rs = np.random.RandomState(3)
    cb = rs.standard_normal((8, 1024, 128)).astype(np.float32)
    lat = rs.standard_normal((32, 128, 900)).astype(np.float32)
    lat[:, :, 700:] = 0.0                                    # zero padding tail as in the reference's padded clips
    cbd, latd = torch.from_numpy(cb).to(cuda), torch.from_numpy(lat).to(cuda)
    codes = ops.rvq_encode(latd, cbd)
    assert codes.shape == (32, 8, 900) and codes.dtype == torch.int64 and int(codes.min()) >= 0 and int(codes.max()) < 1024
    sub = slice(0, 2)
    assert np.array_equal(codes[sub].cpu().numpy(), rvq_oracle.encode(lat[sub], cb))
    # size-independent properties: prefix property (stage q only depends on stages < q), determinism, decode linearity
    c4 = ops.rvq_encode(latd, cbd[:4].contiguous())
    assert torch.equal(c4, codes[:, :4])
    assert torch.equal(ops.rvq_encode(latd, cbd), codes)
    full = ops.rvq_decode(codes, cbd)
    parts = ops.rvq_decode(codes[:, :4].contiguous(), cbd[:4].contiguous()).double() + ops.rvq_decode(codes[:, 4:].contiguous(), cbd[4:].contiguous()).double()
    assert (full.double() - parts).abs().max() < 1e-4
    # each stage picks the nearest code: no other code of that stage is closer to the stage's residual (fp64 audit on a sample)
    r = latd[:1, :, :64].double().permute(0, 2, 1).reshape(-1, 128)
    for q in range(8):
        e = cbd[q].double()
        d2 = ((r[:, None, :] - e[None]) ** 2).sum(-1)
        pick = codes[:1, q, :64].reshape(-1)
        assert (d2.gather(1, pick[:, None])[:, 0] <= d2.min(1).values * (1 + 1e-5) + 1e-6).all()
        r = r - e[pick]
    for T in (1, 31, 129):                                   # ragged lengths / partial tiles
        c = torch.randint(0, 1024, (3, 8, T), device=cuda)
        d = ops.rvq_decode(c, cbd)
        assert np.array_equal(d.cpu().numpy(), rvq_oracle.decode(c.cpu().numpy(), cb))
        c2 = ops.rvq_encode(d, cbd)
        assert np.array_equal(c2.cpu().numpy(), rvq_oracle.encode(d.cpu().numpy(), cb))
    x = torch.randint(0, 1024, (4, 8, 100), device=cuda)
    assert np.array_equal(ops.codes_affine(x).cpu().numpy(), rvq_oracle.codes_affine(x.cpu().numpy()))
    assert torch.equal(ops.codes_affine_inv(ops.codes_affine(x)), x)
