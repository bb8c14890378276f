"""Generates tests/golden/*.npz by running the UNMODIFIED reference (a checkout of the original project, named by
$PROMPT_TTS_REFERENCE and imported with the diffusers-0.15 shim of oracle/diffusers_shim first on sys.path) and transformers'
restatement of encodec (RVQ and SEANet).  The tests read the stored vectors and need neither the reference nor transformers:

    PROMPT_TTS_REFERENCE=<reference checkout> python oracle/make_golden.py
    python oracle/make_golden.py seanet | transformers        (one set only; transformers needed, the reference not)

TEST INFRASTRUCTURE ONLY.  The vectors pin oracle/ref_model.py and oracle/rvq_oracle.c (tests/test_oracle.py)."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "diffusers_shim"))
sys.path.insert(1, HERE)
sys.path.insert(2, os.path.join(ROOT, "tests"))
OUT = os.path.join(ROOT, "tests", "golden")


def denoiser(cfg_name, B, T, seed):
    sys.path.insert(1, os.environ["PROMPT_TTS_REFERENCE"])
    import ref_model
    from tts.models import TTSSingleSpeaker          # the reference's own module tree
    from diffusers import DDPMScheduler              # shim: diffusers 0.15 semantics
    from util import synth_inputs
    cfg = json.load(open(os.path.join(ROOT, "configs", cfg_name + ".json")))
    sd = ref_model.random_state_dict(cfg, seed=seed)
    model = TTSSingleSpeaker(cfg)
    missing = model.load_state_dict(sd, strict=True)
    inp = synth_inputs(cfg, B, T, seed=seed + 1)
    sched = DDPMScheduler(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear")   # train.py:32-36
    xt = sched.add_noise(inp["x0"], inp["noise"], inp["t"])                                                     # train.py:96-98
    pred = model(xt, inp["t"], inp["ids"], inp["mask"]).sample                                                  # train.py:100-105
    loss = torch.nn.functional.mse_loss(pred.float(), inp["noise"].float())                                     # train.py:107
    loss.backward()
    grads = {k: p.grad for k, p in model.named_parameters()}
    out = dict(x0=inp["x0"].numpy(), noise=inp["noise"].numpy(), t=inp["t"].numpy(), ids=inp["ids"].numpy(), mask=inp["mask"].numpy(),
               xt=xt.numpy(), pred=pred.detach().numpy(), loss=np.float64(loss.item()), seed=np.int64(seed),
               weight_checksum=np.float64(sum(float(v.double().sum()) for v in sd.values())))
    names = sorted(grads)
    out["grad_names"] = np.array(names)
    out["grad_norms"] = np.array([0.0 if grads[k] is None else float(grads[k].double().norm()) for k in names])
    for k in ["unet.conv_in.weight", "unet.conv_out.weight", "unet.time_embedding.linear_1.bias", "text_encoder.transformer_blocks.0.norm1.weight",
              "unet.mid_block.attentions.0.transformer_blocks.0.attn2.to_q.weight", "unet.down_blocks.0.resnets.0.time_emb_proj.bias"]:
        out["grad::" + k] = grads[k].numpy()
    # one DDPM sampling step of the shim scheduler (N1 row): pins oracle ddpm_step
    sched.set_timesteps(100)
    g = torch.Generator().manual_seed(7)
    nz = torch.randn(pred.shape, generator=g)
    out["ddpm_t"] = np.int64(990)
    out["ddpm_noise"] = nz.numpy()
    out["ddpm_prev"] = sched.step(pred.detach(), 990, xt, noise=nz).numpy()
    np.savez_compressed(os.path.join(OUT, f"denoiser_{cfg_name}.npz"), **out)
    print("wrote denoiser", cfg_name, "loss", loss.item(), "params", sum(p.numel() for p in model.parameters()))


def rvq_codebooks(seed, grid):
    rs = np.random.RandomState(seed)
    if grid:
        return (rs.randint(-32, 33, size=(8, 1024, 128)) / 16.0).astype(np.float32)
    return rs.standard_normal((8, 1024, 128)).astype(np.float32)


def rvq_latents(seed, B, T, grid):
    rs = np.random.RandomState(seed + 100)
    if grid:
        return (rs.randint(-64, 65, size=(B, 128, T)) / 16.0).astype(np.float32)
    return rs.standard_normal((B, 128, T)).astype(np.float32)


def rvq(name, seed, B, T, grid):
    from transformers import EncodecConfig
    from transformers.models.encodec.modeling_encodec import EncodecResidualVectorQuantizer
    cb, lat = rvq_codebooks(seed, grid), rvq_latents(seed, B, T, grid)
    q = EncodecResidualVectorQuantizer(EncodecConfig())          # 24 kHz defaults: 1024 x 128, 75 fps
    for i in range(8):
        q.layers[i].codebook.embed.copy_(torch.from_numpy(cb[i]))
    codes = q.encode(torch.from_numpy(lat), 6.0)                 # 6 kbps -> 8 quantizers; [8, B, T]
    dec = q.decode(codes).numpy()                                # [B, 128, T]
    codes = codes.permute(1, 0, 2).numpy()                       # reference layout [B, 8, T] (generate_code.py:48)
    np.savez_compressed(os.path.join(OUT, f"rvq_{name}.npz"), seed=np.int64(seed), B=np.int64(B), T=np.int64(T), grid=np.int64(grid),
                        codes=codes.astype(np.int16), dec_slice=dec[:, :, : min(T, 4)].copy(), dec_sum=np.float64(dec.astype(np.float64).sum()),
                        dec_abs_sum=np.float64(np.abs(dec.astype(np.float64)).sum()))
    print("wrote rvq", name, codes.shape)


def seanet():
    """EnCodec SEANet encoder / decoder: transformers' EncodecModel (the installed restatement of encodec 0.1.1; the reference's
    generate_code.py:48 / decode_codec.py:16 run encodec's modules) on the seeded weights of seanet_oracle.make_weights.
    The weights are not stored (60 MB at full width): the tests rebuild them from the seed."""
    import seanet_oracle as so
    out = {}
    for name, cfg, seed, B, S in (("tiny", so.CFG_TINY, 21, 2, 3203), ("k24", so.CFG_24KHZ, 22, 1, 3040)):
        P = so.make_weights(cfg, seed)
        m = so.to_transformers_model(P, cfg)
        wav = (np.random.default_rng(seed).standard_normal((B, 1, S)) * 0.3).astype(np.float32)
        with torch.no_grad():
            lat = m.encoder(torch.from_numpy(wav)).numpy()
            rec = m.decoder(torch.from_numpy(lat)).numpy()
        out.update({f"{name}_seed": np.int64(seed), f"{name}_wav": wav, f"{name}_lat": lat, f"{name}_out": rec})
        print("seanet", name, lat.shape, rec.shape)
    np.savez_compressed(os.path.join(OUT, "seanet_golden.npz"), **out)


# (config, samples) of the SEANet stacks tests/test_seanet_host.py pins seanet_oracle on: weights make_weights(cfg, 3), input
# rng(5).standard_normal((2, 1, samples)) * 0.3
def seanet_pin_variants():
    import seanet_oracle as so
    return ((so.CFG_TINY, 3203), (so.CFG_24KHZ, 3520),
            (dict(so.CFG_TINY, use_causal_conv=False), 3333),           # the asymmetric padding of ME:159-163 / ME:203-204
            (dict(so.CFG_TINY, use_conv_shortcut=False), 2900),         # encodec's true_skip
            (dict(so.CFG_TINY, pad_mode="constant"), 3001),
            (dict(so.CFG_TINY, num_residual_layers=2, dilation_growth_rate=3), 3200))


def seanet_pin_input(S):
    return (np.random.default_rng(5).standard_normal((2, 1, S)) * 0.3).astype(np.float32)


def rvq_full_batch():
    """One complete reference batch (32 clips x 900 frames, generate_code.py:29-34,94-96): Gaussian codebooks and latents, the
    tails of the last 12 clips zero-padded."""
    rs = np.random.RandomState(11)
    cb = rs.standard_normal((8, 1024, 128)).astype(np.float32)
    lat = rs.standard_normal((32, 128, 900)).astype(np.float32)
    lat[20:, :, 650:] = 0.0
    return cb, lat


def transformers_refs():
    """What transformers computes for the tests that pin the oracles and the RVQ kernels against it:
    seanet_transformers.npz -- encoder latents and decoder output (decoder fed transformers' latents) of every
    seanet_pin_variants() stack, with the config each was made with, and the 24 kHz model's encoder / decoder parameter table;
    rvq_full_batch.npz -- codes of encodec's quantiser on rvq_full_batch() at 6 kbps and the SHA-256 of the bytes of its decode of
    those codes (the embedding sum is compared bit for bit; 15 MB of it would not fit the repository)."""
    import hashlib
    import seanet_oracle as so
    from transformers import EncodecConfig, EncodecModel
    from transformers.models.encodec.modeling_encodec import EncodecResidualVectorQuantizer
    out = {}
    for i, (cfg, S) in enumerate(seanet_pin_variants()):
        m = so.to_transformers_model(so.make_weights(cfg, 3), cfg)
        with torch.no_grad():
            lat = m.encoder(torch.from_numpy(seanet_pin_input(S))).numpy()
            wav = m.decoder(torch.from_numpy(lat)).numpy()
        out.update({f"v{i}_cfg": np.array(json.dumps(cfg)), f"v{i}_S": np.int64(S), f"v{i}_lat": lat, f"v{i}_wav": wav})
    sd = EncodecModel(EncodecConfig()).state_dict()
    out["param_shapes_24khz"] = np.array(json.dumps({k: list(v.shape) for k, v in sd.items() if k.startswith(("encoder.", "decoder."))}))
    np.savez_compressed(os.path.join(OUT, "seanet_transformers.npz"), **out)
    cb, lat = rvq_full_batch()
    q = EncodecResidualVectorQuantizer(EncodecConfig())
    with torch.no_grad():
        for i in range(8):
            q.layers[i].codebook.embed.copy_(torch.from_numpy(cb[i]))
        codes = q.encode(torch.from_numpy(lat), 6.0)                         # [8, B, T]
        dec = np.ascontiguousarray(q.decode(codes).numpy())                  # [B, 128, T] fp32
    np.savez_compressed(os.path.join(OUT, "rvq_full_batch.npz"), codes=codes.permute(1, 0, 2).numpy().astype(np.uint16),
                        dec_sha256=np.array(hashlib.sha256(dec.tobytes()).hexdigest()))
    print("wrote seanet_transformers, rvq_full_batch")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if sys.argv[1:] == ["seanet"]:
        seanet()
        sys.exit(0)
    if sys.argv[1:] == ["transformers"]:
        transformers_refs()
        sys.exit(0)
    denoiser("tiny", 2, 16, 0)
    denoiser("tiny3", 2, 32, 1)
    rvq("grid", 0, 3, 77, True)
    rvq("gauss", 1, 2, 150, False)
    seanet()
    transformers_refs()
