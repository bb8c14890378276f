"""GPU: the PUBLIC forward of every module class of the hot path, called standalone with the reference's signature (SURVEY 4 ii /
8b), forward + input gradients + every parameter gradient against the oracle's restatement of the same reference function
(oracle/ref_model.py).  Real widths (320 / 640 channels, head dims 40 / 80, 768-d text context, GroupNorm groups of 10 / 20 / 30).
Bar: 2e-2 relative on outputs, input gradients and the global parameter-gradient vector (bf16 compute)."""
import pytest
import torch
import torch.nn.functional as F

import ref_model
import training_oracle as to
from util import load_model, rel, synth_inputs

pytestmark = pytest.mark.gpu
TOL = 2e-2


def _sd(module, prefix="m"):
    return {f"{prefix}.{k}": v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in module.state_dict().items()}


def _check(module, outs, ref_outs, inputs, ref_inputs, sd, prefix="m"):
    outs = outs if isinstance(outs, (tuple, list)) else [outs]
    ref_outs = ref_outs if isinstance(ref_outs, (tuple, list)) else [ref_outs]
    assert len(outs) == len(ref_outs)
    g = torch.Generator(device="cuda").manual_seed(99)
    loss = ref_loss = 0.0
    for o, r in zip(outs, ref_outs):
        assert o.shape == r.shape and o.dtype == torch.float32, (o.shape, r.shape, o.dtype)
        assert rel(o, r) < TOL, ("output", rel(o, r))
        w = torch.randn(r.shape, device="cuda", generator=g)
        loss = loss + (o * w).sum()
        ref_loss = ref_loss + (r * w).sum()
    loss.backward()
    ref_loss.backward()
    for x, xr in zip(inputs, ref_inputs):
        if xr.grad is not None:
            assert x.grad is not None and rel(x.grad, xr.grad) < TOL, ("input grad", rel(x.grad, xr.grad))
    ours, refs = [], []
    for k, p in module.named_parameters():
        gr = sd[f"{prefix}.{k}"].grad
        if gr is None or gr.abs().max() == 0:                   # dead proj_out
            assert p.grad is None or p.grad.abs().max() == 0, k
            continue
        assert p.grad is not None and p.grad.shape == p.shape, k
        assert rel(p.grad, gr) < 6e-2, (k, rel(p.grad, gr))
        ours.append(p.grad.flatten())
        refs.append(gr.flatten())
    e = rel(torch.cat(ours), torch.cat(refs))
    assert e < TOL, ("global parameter gradient", e)
    return e


def _inputs(*shapes, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    xs = [torch.randn(s, device="cuda", generator=g).requires_grad_(True) for s in shapes]
    return xs, [x.detach().clone().requires_grad_(True) for x in xs]


@pytest.mark.parametrize("cin,cout", [(320, 320), (320, 640), (960, 640)])
def test_resnet_block_forward(cuda, cin, cout):
    """ResnetBlock1D.forward(input_tensor, temb)  (reference tts/ldm/resnet.py:231-283)"""
    from prompt_tts_b200.ldm.resnet import ResnetBlock1D
    torch.manual_seed(0)
    m = ResnetBlock1D(in_channels=cin, out_channels=cout, temb_channels=1280, eps=1e-5, groups=32).cuda()
    (x, t), (xr, tr) = _inputs((3, cin, 188), (3, 1280))
    sd = _sd(m)
    _check(m, m(x, t), ref_model.resnet_block(sd, "m", xr, tr), [x, t], [xr, tr], sd)


def test_up_down_sample_forward(cuda):
    """Upsample1D.forward(x, output_size) / Downsample1D.forward(hidden_states)  (resnet.py:36-49, 87-96)"""
    from prompt_tts_b200.ldm.resnet import Downsample1D, Upsample1D
    torch.manual_seed(0)
    up = Upsample1D(320, use_conv=True, out_channels=320).cuda()
    (x,), (xr,) = _inputs((2, 320, 94))
    sd = _sd(up)
    ref = F.conv1d(F.interpolate(xr, scale_factor=2.0, mode="nearest"), sd["m.conv.weight"], sd["m.conv.bias"], padding=1)
    _check(up, up(x, output_size=188), ref, [x], [xr], sd)
    down = Downsample1D(320, use_conv=True, out_channels=320, padding=1, name="op").cuda()
    (x,), (xr,) = _inputs((2, 320, 187), seed=1)            # odd length: floor((L - 1) / 2) + 1 output frames
    sd = _sd(down)
    ref = F.conv1d(xr, sd["m.conv.weight"], sd["m.conv.bias"], stride=2, padding=1)
    _check(down, down(x), ref, [x], [xr], sd)


@pytest.mark.parametrize("C", [320, 640])
def test_transformer_1d_forward(cuda, C):
    """Transformer1DModel.forward(hidden_states, encoder_hidden_states, ..., return_dict)  (transformer_1d.py:199-310)"""
    from prompt_tts_b200.ldm.transformer_1d import Transformer1DModel, Transformer1DModelOutput
    torch.manual_seed(0)
    m = Transformer1DModel(8, C // 8, in_channels=C, num_layers=1, cross_attention_dim=768, norm_num_groups=32).cuda()
    (x, e), (xr, er) = _inputs((2, C, 188), (2, 77, 768))
    sd = _sd(m)
    out = m(x, encoder_hidden_states=e)
    assert isinstance(out, Transformer1DModelOutput)
    tup = m(x.detach(), encoder_hidden_states=e.detach(), return_dict=False)
    # (two runs are not bit-identical: GroupNorm statistics are accumulated with fp32 atomics, whose order can move a bf16 rounding)
    assert isinstance(tup, tuple) and rel(tup[0], out.sample.detach()) < 2e-3
    _check(m, out.sample, ref_model.transformer_1d(sd, "m", xr, er, 8), [x, e], [xr, er], sd)
    assert m.proj_out.weight.grad is None or m.proj_out.weight.grad.abs().max() == 0      # constructed, never applied (:190 vs :275-279)


def _ref_down(sd, xr, tr, er, n, attn, down):
    h, outs = xr, []
    for j in range(n):
        h = ref_model.resnet_block(sd, f"m.resnets.{j}", h, tr)
        if attn:
            h = ref_model.transformer_1d(sd, f"m.attentions.{j}", h, er, 8)
        outs.append(h)
    if down:
        h = F.conv1d(h, sd["m.downsamplers.0.conv.weight"], sd["m.downsamplers.0.conv.bias"], stride=2, padding=1)
        outs.append(h)
    return [h] + outs


def test_down_blocks_forward(cuda):
    """CrossAttnDownBlock1D.forward / DownBlock1D.forward -> (hidden_states, output_states)  (unet_blocks.py:257-281, 359-408)"""
    from prompt_tts_b200.ldm.unet_blocks import get_down_block
    torch.manual_seed(0)
    kw = dict(temb_channels=1280, resnet_eps=1e-5, resnet_act_fn="silu", attn_num_head_channels=8, resnet_groups=32,
              cross_attention_dim=768, downsample_padding=1)
    m = get_down_block("CrossAttnDownBlock1D", num_layers=2, in_channels=320, out_channels=640, add_downsample=True, **kw).cuda()
    (x, t, e), (xr, tr, er) = _inputs((2, 320, 96), (2, 1280), (2, 50, 768))
    sd = _sd(m)
    h, states = m(x, t, encoder_hidden_states=e)
    assert isinstance(states, tuple) and len(states) == 3 and torch.equal(h, states[-1])
    _check(m, [h, *states], _ref_down(sd, xr, tr, er, 2, True, True), [x, t, e], [xr, tr, er], sd)
    m = get_down_block("UNetResDownBlock1D", num_layers=2, in_channels=640, out_channels=640, add_downsample=False, **kw).cuda()
    (x, t), (xr, tr) = _inputs((2, 640, 48), (2, 1280), seed=2)
    sd = _sd(m)
    h, states = m(x, t)
    assert len(states) == 2
    _check(m, [h, *states], _ref_down(sd, xr, tr, None, 2, False, False), [x, t], [xr, tr], sd)


def test_mid_and_up_blocks_forward(cuda):
    """UNetMidBlock1DCrossAttn.forward, UpBlock1D.forward, CrossAttnUpBlock1D.forward  (unet_blocks.py:603-620, 179-202, 482-529)"""
    from prompt_tts_b200.ldm.unet_blocks import UNetMidBlock1DCrossAttn, get_up_block
    torch.manual_seed(0)
    m = UNetMidBlock1DCrossAttn(in_channels=640, temb_channels=1280, resnet_eps=1e-5, resnet_act_fn="silu", attn_num_head_channels=8,
                                resnet_groups=32, cross_attention_dim=768).cuda()
    (x, t, e), (xr, tr, er) = _inputs((2, 640, 48), (2, 1280), (2, 50, 768))
    sd = _sd(m)
    ref = ref_model.resnet_block(sd, "m.resnets.0", xr, tr)
    ref = ref_model.resnet_block(sd, "m.resnets.1", ref_model.transformer_1d(sd, "m.attentions.0", ref, er, 8), tr)
    _check(m, m(x, t, encoder_hidden_states=e), ref, [x, t, e], [xr, tr, er], sd)

    kw = dict(temb_channels=1280, resnet_eps=1e-5, resnet_act_fn="silu", attn_num_head_channels=8, resnet_groups=32, cross_attention_dim=768)
    for typ, attn in (("UpBlock1D", False), ("CrossAttnUpBlock1D", True)):
        m = get_up_block(typ, num_layers=3, in_channels=320, out_channels=640, prev_output_channel=640, add_upsample=True, **kw).cuda()
        # skips are popped from the END of the tuple: channels 640, 640, 320 in consumption order
        (x, t, e, s0, s1, s2), (xr, tr, er, r0, r1, r2) = _inputs((2, 640, 48), (2, 1280), (2, 50, 768), (2, 320, 48), (2, 640, 48), (2, 640, 48), seed=3)
        sd = _sd(m)
        if attn:
            out = m(x, (s0, s1, s2), t, encoder_hidden_states=e)
        else:
            out = m(x, (s0, s1, s2), t, upsample_size=96)
        h = xr
        for j, sk in enumerate((r2, r1, r0)):
            h = ref_model.resnet_block(sd, f"m.resnets.{j}", torch.cat([h, sk], 1), tr)
            if attn:
                h = ref_model.transformer_1d(sd, f"m.attentions.{j}", h, er, 8)
        h = F.conv1d(F.interpolate(h, scale_factor=2.0, mode="nearest"), sd["m.upsamplers.0.conv.weight"], sd["m.upsamplers.0.conv.bias"], padding=1)
        ins, rins = ([x, t, e, s0, s1, s2], [xr, tr, er, r0, r1, r2]) if attn else ([x, t, s0, s1, s2], [xr, tr, r0, r1, r2])
        _check(m, out, h, ins, rins, sd)


def test_text_encoder_and_unet_forward(cuda):
    """TextEncoder.forward(input_ids, attention_mask) and Unet1DConditionModel.forward(sample, timestep, encoder_hidden_states, ...)
    called on their own (models.py:106-120, unet_1d_condition.py:553-739), timestep as tensor / 0-d tensor / int."""
    cfg, model = load_model("mid", cuda, train=True)
    inp = synth_inputs(cfg, 2, 64, seed=5, device="cuda")
    sd = to.oracle_params(model)
    enc = model.text_encoder(inp["ids"], inp["mask"])
    ref_enc = ref_model.text_encoder(sd, cfg, inp["ids"])
    assert rel(enc, ref_enc) < TOL
    x = inp["x0"].clone().requires_grad_(True)
    e = ref_enc.detach().clone().requires_grad_(True)
    out = model.unet(x, inp["t"], encoder_hidden_states=e, attention_mask=inp["mask"]).sample
    xr, er = x.detach().clone().requires_grad_(True), e.detach().clone().requires_grad_(True)
    ref = ref_model.unet(sd, cfg, xr, inp["t"], er)
    assert rel(out, ref) < TOL
    w = torch.randn_like(ref)
    (out * w).sum().backward()
    (ref * w).sum().backward()
    assert rel(e.grad, er.grad) < TOL, rel(e.grad, er.grad)
    with torch.no_grad():
        t0 = int(inp["t"][0])
        a = model.unet(inp["x0"][:1], t0, encoder_hidden_states=ref_enc[:1].detach(), return_dict=False)[0]
        b = model.unet(inp["x0"][:1], torch.tensor(t0, device="cuda"), encoder_hidden_states=ref_enc[:1].detach()).sample
    assert rel(a, b) < 2e-3
