"""GPU: classifier-free guidance.  The three entry points bit for bit against torch, the null-context shortcut of a transformer
block bit for bit against the product's own unguided block, one guided denoiser forward and the guided DDPM / DDIM / DPM-Solver++
loops against an fp32 oracle (oracle/ref_model.py denoiser on the text encoding and on zeros, eps_u + w (eps_c - eps_u), the
shim's step), and condition dropout in the train step and in TTSSingleSpeaker.forward against the oracle with the text encoding
selected by the keep mask."""
import pytest
import torch

import sampling_oracle as so
from util import rel, synth_inputs

pytestmark = pytest.mark.gpu
TOL = 2e-2


# ---------------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("w", [1.0, 1.5, 3.0, 7.5, 12.345678])
def test_cfg_combine_matches_torch_bitwise(cuda, w):
    from prompt_tts_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(1)
    n = 3 * 8 * 40 + 5
    eps2 = torch.randn(2, n, device=cuda, generator=g) * 3
    c, u = eps2[0].clone(), eps2[1].clone()
    want = u + w * (c - u)
    out = torch.empty(n, device=cuda)
    ops.call("cfg_combine", ops._p(eps2), ops._p(out), n, w, ops._stream())
    assert torch.equal(out, want)
    ops.call("cfg_combine", ops._p(eps2), ops._p(eps2), n, w, ops._stream())        # out aliasing the conditional half
    assert torch.equal(eps2[0], want) and torch.equal(eps2[1], u)


def test_cond_select_matches_where(cuda):
    from prompt_tts_b200 import ops
    B, L, D = 6, 24, 64
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(B, L, D, device=cuda, generator=g).to(torch.bfloat16)
    keep = torch.tensor([1, 0, 1, 0, 0, 1], dtype=torch.bool, device=cuda)
    x[1, 3, 5] = float("nan")
    x[3, 0, 0] = float("inf")
    x[4, 7] = -float("inf")
    x[2, 1, 1] = float("inf")                 # kept: passes through
    want = torch.where(keep[:, None, None], x, torch.zeros_like(x))
    y = torch.full_like(x, 7.0)
    ops.call("cond_select_bf16", ops._p(x), ops._p(keep), ops._p(y), B, L * D, ops._stream())
    assert torch.equal(y, want) and torch.isfinite(y[~keep]).all()
    k8 = torch.tensor([3, 0, 255, 0, 0, 1], dtype=torch.uint8, device=cuda)     # any nonzero byte keeps
    ops.call("cond_select_bf16", ops._p(x), ops._p(k8), ops._p(x), B, L * D, ops._stream())     # in place
    assert torch.equal(x, want)


@pytest.mark.parametrize("rows,K,C", [(96, 64, 64), (376, 320, 320), (33, 640, 640)])
def test_rows_add_bias_is_the_gemm_with_a_zero_operand(cuda, rows, K, C):
    from prompt_tts_b200 import engine as E
    from prompt_tts_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(rows)
    w = torch.randn(C, K, device=cuda, generator=g) * 0.05
    b = torch.randn(C, device=cuda, generator=g)
    b[:4] = torch.tensor([0.0, -0.0, 1e-30, -3.0])
    res = (torch.randn(rows, C, device=cuda, generator=g) * 4).to(torch.bfloat16)
    tape = E.Tape(E.PackCache(), recording=False)
    want = E.linear(tape, E.Var(torch.zeros(rows, K, dtype=torch.bfloat16, device=cuda)), [w], [b], residual=E.Var(res)).data
    y = torch.empty_like(res)
    ops.call("rows_add_bias_bf16", ops._p(res), ops._p(b), ops._p(y), rows, C, ops._stream())
    assert torch.equal(y, want)
    ops.call("rows_add_bias_bf16", ops._p(res), ops._p(b), ops._p(res), rows, C, ops._stream())     # in place
    assert torch.equal(res, want)


# ---------------------------------------------------------------------------------------------------------------- shortcut
@pytest.mark.parametrize("dim,ctx,Lk", [(64, 64, 24), (320, 768, 64), (640, 768, 77)])
@pytest.mark.parametrize("B", [1, 3])
def test_block_null_context_shortcut_is_exact(cuda, dim, ctx, Lk, B):
    """A BasicTransformerBlock at the `tiny` / `mid` widths (8 heads, as the UNet builds them).  Guided forward at 2B rows: the
    conditional rows equal the product's unguided block at batch B with the text context, the unconditional rows the same block
    with an all-zero context, bit for bit."""
    from prompt_tts_b200 import engine as E
    from prompt_tts_b200.ldm.attention import BasicTransformerBlock
    torch.manual_seed(dim + B)
    blk = BasicTransformerBlock(dim, 8, dim // 8, cross_attention_dim=ctx).to(cuda)
    with torch.no_grad():                                    # non-trivial LayerNorm affine and to_out bias
        for p in blk.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.3)
    L = 94
    g = torch.Generator(device="cuda").manual_seed(B)
    h = torch.randn(2 * B, L, dim, device=cuda, generator=g).to(torch.bfloat16)
    enc = torch.randn(B, Lk, ctx, device=cuda, generator=g).to(torch.bfloat16)
    cache = E.get_cache(blk)

    def run(hd, ed, cond_rows=None):
        tape = E.Tape(cache, recording=False)
        tape.cond_rows = cond_rows
        return blk._fwd(tape, E.Var(hd.clone(), needs_grad=False), E.Var(ed.clone(), needs_grad=False)).data

    guided = run(h, enc, cond_rows=B)
    cond = run(h[:B], enc)
    uncond = run(h[B:], torch.zeros_like(enc))
    d_c = (guided[:B].float() - cond.float()).abs().max().item()
    d_u = (guided[B:].float() - uncond.float()).abs().max().item()
    print(f"\n[block {dim}/{ctx} B={B}] max |guided - unguided|: conditional rows {d_c:.3g}, unconditional rows {d_u:.3g}")
    assert torch.equal(guided[:B], cond)
    assert torch.equal(guided[B:], uncond)
    with pytest.raises(AssertionError, match="inference-only"):
        tape = E.Tape(cache, recording=True)
        tape.cond_rows = B
        blk._fwd(tape, E.Var(h.clone()), E.Var(enc.clone()))


# ---------------------------------------------------------------------------------------------------------------- one forward
@pytest.mark.parametrize("cfg_name", ["tiny", "tiny3", "mid", "1d_config"])
def test_guided_forward_matches_oracle(cuda, cfg_name):
    import ref_model
    from prompt_tts_b200 import engine as E
    cfg, model = so.load_model(cfg_name, cuda)
    B, T = 1, 752
    inp = synth_inputs(cfg, B, T, seed=4, device=cuda)
    x = inp["noise"]
    t = torch.full((2 * B,), 600, dtype=torch.int64, device=cuda)
    with torch.no_grad():
        tape = E.Tape(E.get_cache(model), recording=False)
        tape.kv_cache = {}
        enc = model.text_encoder._fwd(tape, inp["ids"])
        tape.cond_rows = B
        eps2, _ = model.unet._fwd(tape, torch.cat([x, x]).contiguous(), t, enc)
        sd = {k: v.detach().float() for k, v in model.state_dict().items()}
        enc_r = ref_model.text_encoder(sd, cfg, inp["ids"])
        want_c = ref_model.unet(sd, cfg, x, t[:B], enc_r)
        want_u = ref_model.unet(sd, cfg, x, t[:B], torch.zeros_like(enc_r))
    e_c, e_u = rel(eps2[:B], want_c), rel(eps2[B:], want_u)
    print(f"\n[{cfg_name} guided forward B={B} T={T}] conditional {e_c:.2e}, unconditional {e_u:.2e} (halves differ by "
          f"{rel(want_u, want_c):.2e})")
    assert e_c < TOL and e_u < TOL, (e_c, e_u)


# ---------------------------------------------------------------------------------------------------------------- loops
KINDS = [("ddpm", None), ("ddim", 0.0), ("ddim", 1.0), ("dpm", None)]


@pytest.fixture(scope="module")
def tiny(cuda):
    return so.load_model("tiny", cuda)


@pytest.mark.parametrize("kind,eta", KINDS)
def test_guided_loop_matches_oracle(cuda, tiny, kind, eta):
    cfg, model = tiny
    B, T, n_infer, w = 2, 16, 5, 3.0
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 5, cuda)
    outs = {gr: so.make_sampler(model, kind, eta, n_infer, use_graph=gr).sample(inp["ids"], T, x_T=x_T, noises=noises, guidance_scale=w)
            for gr in (False, True)}
    assert outs[True].shape == x_T.shape and outs[True].is_contiguous()
    # GroupNorm statistics are accumulated with fp32 atomics (order not fixed), so two runs agree to rounding, not bit for bit
    assert rel(outs[False], outs[True]) < 1e-3, "graph replay must reproduce the eager loop"
    x = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=w)
    unguided = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=1.0)
    # guidance multiplies a per-call error of the denoiser by about w: the bar is what the fp32 oracle loop makes of the 2e-2
    # per-call bar on each of eps_c and eps_u
    bound = rel(so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=w, eps_err=TOL, err_seed=23), x)
    e = {gr: rel(outs[gr], x) for gr in (False, True)}
    print(f"\n[guided {kind} eta={eta} tiny w={w}, {n_infer} steps] rel err vs fp32 oracle loop: graph {e[True]:.2e}, eager "
          f"{e[False]:.2e} (bound {bound:.2e}; guided vs unguided oracle {rel(x, unguided):.2e})")
    assert e[True] < bound and e[False] < bound, (e, bound)


@pytest.mark.parametrize("kind,eta", KINDS)
def test_guided_loop_prompt_and_codes(cuda, tiny, kind, eta):
    cfg, model = tiny
    B, T, P, n_infer, w = 2, 16, 6, 4, 3.0
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 6, cuda)
    prompt = inp["x0"][..., :P].contiguous()
    smp = so.make_sampler(model, kind, eta, n_infer)
    x = smp.sample(inp["ids"], T, prompt=prompt, seed=3, guidance_scale=w)
    assert torch.equal(x[..., :P], prompt), "the prompt frames must come out clean"
    assert torch.isfinite(x).all()
    codes = smp.sample(inp["ids"], T, prompt=prompt, seed=3, return_codes=True, guidance_scale=w)
    assert torch.equal(codes, torch.clamp(torch.round((x + 1) * 511.5), 0, 1023).to(torch.int64))
    g = torch.Generator(device="cuda").manual_seed(12)
    pn = torch.randn(n_infer, B, cfg["in_channels"], P, device=cuda, generator=g)
    got = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, prompt=prompt, prompt_noise=pn, guidance_scale=w)
    want = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=w, prompt=prompt, prompt_noise=pn)
    bound = rel(so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=w, prompt=prompt, prompt_noise=pn,
                               eps_err=TOL, err_seed=23), want)
    print(f"\n[guided {kind} eta={eta} + prompt] rel err {rel(got, want):.2e} (bound {bound:.2e})")
    assert torch.equal(got[..., :P], want[..., :P])
    assert rel(got, want) < bound


@pytest.mark.parametrize("kind,eta", [("ddpm", None), ("dpm", None)])
def test_guided_loop_batch_one(cuda, tiny, kind, eta):
    cfg, model = tiny
    B, T, n_infer, w = 1, 32, 5, 4.0
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 7, cuda)
    got = so.make_sampler(model, kind, eta, n_infer).sample(inp["ids"], T, x_T=x_T, noises=noises, guidance_scale=w)
    want = so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=w)
    bound = rel(so.oracle_loop(model, cfg, kind, eta, n_infer, inp["ids"], x_T, noises, w=w, eps_err=TOL, err_seed=23), want)
    print(f"\n[guided {kind} B=1 w={w}] rel err {rel(got, want):.2e} (bound {bound:.2e})")
    assert rel(got, want) < bound


def test_guided_loop_prompt_tokens(cuda, tiny):
    """prompt tokens extend the conditional rows' context only; the result differs from the text-only guided run"""
    cfg, model = tiny
    B, T, n_infer = 2, 16, 3
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 8, cuda)
    toks = torch.randn(B, 9, cfg["cross_attention_dim"], device=cuda)
    smp = so.make_sampler(model, "dpm", None, n_infer)
    a = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, prompt_tokens=toks, guidance_scale=2.0)
    b = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, guidance_scale=2.0)
    assert torch.isfinite(a).all() and rel(a, b) > 1e-3


def test_guidance_one_is_the_unguided_loop(cuda, tiny):
    """guidance_scale = 1 allocates batch-B buffers only (no unconditional forward) and gives the unguided result"""
    from prompt_tts_b200 import _lib
    cfg, model = tiny
    B, T, n_infer = 2, 16, 4
    inp, x_T, noises = so.case(cfg, B, T, n_infer, 9, cuda)
    smp = so.make_sampler(model, "ddim", 0.0, n_infer)
    smp.sample(inp["ids"], T, x_T=x_T, noises=noises)          # first-use work (weight packs) outside the counted calls
    lib = _lib.lib()
    l0 = lib.pt_launch_count()
    a = smp.sample(inp["ids"], T, x_T=x_T, noises=noises)
    n_default = lib.pt_launch_count() - l0
    assert "x2" not in smp._static and smp._static["x"].shape[0] == B and smp._static["t"].shape[0] == B
    l0 = lib.pt_launch_count()
    b = smp.sample(inp["ids"], T, x_T=x_T, noises=noises, guidance_scale=1.0)
    assert lib.pt_launch_count() - l0 == n_default
    assert "x2" not in smp._static and smp._static["t"].shape[0] == B
    assert rel(a, b) < 1e-3
    smp.sample(inp["ids"], T, x_T=x_T, noises=noises, guidance_scale=1.5)
    assert smp._static["x2"].shape[0] == 2 * B and smp._static["t"].shape[0] == 2 * B and smp._static["eps"].shape[0] == B


# ---------------------------------------------------------------------------------------------------------------- training
def _oracle_train(cfg, model, inp, keep):
    """add_noise, the text encoding selected by keep (zeros where dropped), the UNet, MSE: fp32 autograd"""
    import ref_model
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point() and "inv_freq" not in k) for k, v in model.state_dict().items()}
    xt = ref_model.add_noise(inp["x0"], inp["noise"], inp["t"])
    enc = ref_model.text_encoder(sd, cfg, inp["ids"])
    enc = torch.where(keep.bool()[:, None, None], enc, torch.zeros_like(enc))
    pred = ref_model.unet(sd, cfg, xt, inp["t"], enc)
    loss = torch.nn.functional.mse_loss(pred, inp["noise"])
    loss.backward()
    return xt, loss.detach(), {k: v.grad for k, v in sd.items() if v.requires_grad and v.grad is not None and v.grad.abs().max() > 0}


def _keep(B, dev):
    return (torch.arange(B, device=dev) % 3 != 1)          # mixed: 1, 0, 1, 1, 0, 1, ...


# sizes and the reason for them: test_model_gpu.py (fewer positions per weight-gradient sum and no bf16 path meets 2e-2)
@pytest.mark.parametrize("cfg_name,B,T", [("tiny", 8, 64), ("tiny3", 8, 128), ("mid", 2, 64)])
def test_train_step_condition_dropout_matches_oracle(cuda, cfg_name, B, T):
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model(cfg_name, cuda, train=True)
    inp = synth_inputs(cfg, B, T, seed=1, device=cuda)
    keep = _keep(B, cuda)
    assert keep.any() and not keep.all()
    _, ref_loss, ref_grads = _oracle_train(cfg, model, inp, keep)
    loss = DenoiserTrainStep(model)(inp["x0"], inp["noise"], inp["t"], inp["ids"], inp["mask"], cond_keep=keep)
    torch.cuda.synchronize()
    e_l, e_g = rel(loss, ref_loss), so.grad_err(model, ref_grads)
    print(f"\n[{cfg_name} {B}x{T} condition dropout, keep {keep.int().tolist()}] loss {e_l:.2e} global grad {e_g:.2e}")
    assert e_l < TOL and e_g < TOL, (e_l, e_g)


def test_train_step_all_dropped(cuda):
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 8, 64
    inp = synth_inputs(cfg, B, T, seed=2, device=cuda)
    none = torch.zeros(B, dtype=torch.bool, device=cuda)
    stepper = DenoiserTrainStep(model)
    l1 = float(stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], cond_keep=none))
    named = dict(model.named_parameters())
    cross_kv = [k for k in named if ".attn2.to_k." in k or ".attn2.to_v." in k]
    text = [k for k in named if k.startswith("text_encoder.")]
    assert cross_kv and text
    for k in cross_kv + text:
        g = named[k].grad
        assert g is None or torch.count_nonzero(g) == 0, k
    assert any(named[k].grad is not None and torch.count_nonzero(named[k].grad) > 0 for k in named if k.startswith("unet."))
    other = synth_inputs(cfg, B, T, seed=77, device=cuda)["ids"]
    assert not torch.equal(other, inp["ids"])
    l2 = float(stepper(inp["x0"], inp["noise"], inp["t"], other, cond_keep=none))
    assert abs(l1 - l2) <= 1e-3 * abs(l1), (l1, l2)          # GroupNorm atomics: not bit-reproducible run to run
    # a mixed mask does reach the text encoder
    stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], cond_keep=_keep(B, cuda))
    assert all(named[k].grad is not None and torch.count_nonzero(named[k].grad) > 0 for k in cross_kv)


def test_train_step_all_kept_is_the_default(cuda):
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 8, 64
    inp = synth_inputs(cfg, B, T, seed=3, device=cuda)
    stepper = DenoiserTrainStep(model)
    named = list(model.named_parameters())
    l_none = float(stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"]))
    g_none = torch.cat([p.grad.flatten() for _, p in named if p.grad is not None]).clone()
    l_all = float(stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], cond_keep=torch.ones(B, dtype=torch.uint8, device=cuda)))
    g_all = torch.cat([p.grad.flatten() for _, p in named if p.grad is not None])
    assert abs(l_none - l_all) <= 1e-3 * abs(l_none) and rel(g_all, g_none) < 1e-3


def test_train_step_graph_replays_fresh_masks(cuda):
    """a captured step reads the mask from its static buffer: replays with two masks equal eager steps with the same masks"""
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 8, 64
    inp = synth_inputs(cfg, B, T, seed=4, device=cuda)
    stepper = DenoiserTrainStep(model)
    keep = torch.ones(B, dtype=torch.bool, device=cuda)
    loss = torch.zeros((), device=cuda)
    masks = [_keep(B, cuda), torch.arange(B, device=cuda) % 2 == 0]
    named = list(model.named_parameters())

    def step():
        return stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], loss_out=loss, cond_keep=keep)

    eager = []
    for m in masks:
        keep.copy_(m)
        step()
        torch.cuda.synchronize()
        eager.append((float(loss), torch.cat([p.grad.flatten() for _, p in named if p.grad is not None]).clone()))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for m, (l_e, g_e) in zip(masks, eager):
        keep.copy_(m)
        graph.replay()
        torch.cuda.synchronize()
        g = torch.cat([p.grad.flatten() for _, p in named if p.grad is not None])
        assert abs(float(loss) - l_e) <= 1e-3 * abs(l_e) and rel(g, g_e) < 1e-3
    assert rel(eager[0][1], eager[1][1]) > 1e-3, "the two masks must give different gradients"


def test_model_forward_cond_keep_matches_oracle(cuda):
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 8, 64
    inp = synth_inputs(cfg, B, T, seed=5, device=cuda)
    keep = _keep(B, cuda)
    xt, ref_loss, ref_grads = _oracle_train(cfg, model, inp, keep)
    out = model(xt, inp["t"], inp["ids"], inp["mask"], cond_keep=keep).sample
    loss = torch.nn.functional.mse_loss(out, inp["noise"])
    loss.backward()
    torch.cuda.synchronize()
    e_l, e_g = rel(loss, ref_loss), so.grad_err(model, ref_grads)
    print(f"\n[TTSSingleSpeaker.forward cond_keep, tiny {B}x{T}] loss {e_l:.2e} global grad {e_g:.2e}")
    assert e_l < TOL and e_g < TOL, (e_l, e_g)


def test_bad_cond_keep_raises(cuda):
    from prompt_tts_b200 import _lib
    from prompt_tts_b200.train import DenoiserTrainStep
    cfg, model = so.load_model("tiny", cuda, train=True)
    B, T = 2, 16
    inp = synth_inputs(cfg, B, T, seed=6, device=cuda)
    stepper = DenoiserTrainStep(model)
    for bad in (torch.ones(B + 1, dtype=torch.bool, device=cuda), torch.ones(B, 1, dtype=torch.bool, device=cuda),
                torch.ones(B, dtype=torch.float32, device=cuda), torch.ones(B, dtype=torch.int64, device=cuda),
                torch.ones(B, dtype=torch.bool)):
        with pytest.raises(_lib.PtError, match="cond_keep"):
            stepper(inp["x0"], inp["noise"], inp["t"], inp["ids"], cond_keep=bad)
        with pytest.raises(_lib.PtError, match="cond_keep"):
            model(inp["x0"], inp["t"], inp["ids"], inp["mask"], cond_keep=bad)
