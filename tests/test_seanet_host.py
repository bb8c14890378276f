"""CPU tier for the SEANet row (SURVEY 8f-4): the oracle against transformers' EnCodec modules and the golden vectors, the C ABI
of libpt_seanet.so, and the kernels' index arithmetic through the host-side grid walker (tests/seanet_emul.cpp).

`EmuDriver` below is a TEST double: it hands `prompt_tts_b200.codec.SeanetStack` -- the product's layer sequencing -- the
seanet_core.h bodies compiled for the host, so buffer routing, padding and activation placement are checked here without a
GPU.  The product never constructs it (see test_product_raises_without_gpu)."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import seanet_oracle as so  # noqa: E402
from prompt_tts_b200 import codec  # noqa: E402

EMUL_SO = os.path.join(ROOT, "oracle", "_build", "libseanet_emul.so")


class EmuDriver:
    """numpy memory + the host build of the kernel bodies; NaN-filled allocations so a read of an unwritten element shows."""

    def __init__(self):
        src = [os.path.join(ROOT, "tests", "seanet_emul.cpp"), os.path.join(ROOT, "prompt_tts_b200", "csrc", "seanet", "seanet_core.h")]
        if not os.path.exists(EMUL_SO) or any(os.path.getmtime(s) > os.path.getmtime(EMUL_SO) for s in src):
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
        self.lib = C.CDLL(EMUL_SO)
        ct = {"p": C.c_void_p, "i": C.c_int}
        for name, sig in codec.SIGS.items():
            fn = getattr(self.lib, "emu_sn_" + name)
            fn.argtypes = [ct[c] for c in sig[:-1]]          # same arguments minus the stream
            fn.restype = None
        self.calls = []

    def empty(self, *shape):
        return np.full(shape, np.nan, np.float32)

    def ptr(self, buf):
        return 0 if buf is None else buf.ctypes.data

    def upload(self, a):
        return np.ascontiguousarray(np.asarray(a, np.float32))

    def call(self, name, *args):
        self.calls.append(name)
        getattr(self.lib, "emu_sn_" + name)(*args)


@pytest.fixture(scope="module")
def drv():
    return EmuDriver()


def rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b.astype(np.float64)) / max(np.linalg.norm(b.astype(np.float64)), 1e-30))


# ------------------------------------------------------------------------------------------------ oracle pinning
def test_oracle_matches_transformers_tiny_and_24khz():
    """transformers' EncodecModel on the same weights and input, as stored by oracle/make_golden.py (transformers)."""
    import make_golden as mg
    g = np.load(os.path.join(ROOT, "tests", "golden", "seanet_transformers.npz"))
    variants = mg.seanet_pin_variants()
    assert len(variants) == 6
    for i, (cfg, S) in enumerate(variants):
        assert json.loads(str(g[f"v{i}_cfg"])) == json.loads(json.dumps(cfg)) and int(g[f"v{i}_S"]) == S, (i, "regenerate the golden file")
        P = so.make_weights(cfg, 3)
        x = mg.seanet_pin_input(S)
        lat_ref, wav_ref = g[f"v{i}_lat"], g[f"v{i}_wav"]
        lat = so.encoder(x, P, cfg)
        assert lat.shape == lat_ref.shape == (2, cfg["hidden_size"], -(-S // 320))
        assert rel(lat, lat_ref) < 1e-5
        wav = so.decoder(lat_ref, P, cfg)
        assert wav.shape == wav_ref.shape == (2, 1, 320 * lat.shape[-1])
        assert rel(wav, wav_ref) < 1e-5


def test_oracle_param_table_is_transformers_state_dict():
    """The encoder / decoder tensors of transformers' EncodecModel(EncodecConfig()), as stored by oracle/make_golden.py."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "seanet_transformers.npz"))
    want = {k: tuple(v) for k, v in json.loads(str(g["param_shapes_24khz"])).items()}
    assert so.param_shapes(so.CFG_24KHZ) == want
    # the product's plan names exactly the same tensors
    model_names = []
    for side in ("encoder", "decoder"):
        model_names += codec.SeanetStack(codec.CFG_24KHZ, side, None).param_names()
    assert sorted(model_names) == sorted(want)
    strip = lambda plan: {k: [(i, kind, {a: b for a, b in s.items() if not (kind == "convtr" and a == "dil")}) for i, kind, s in v]
                          for k, v in plan.items()}
    assert strip(codec.layer_plan(codec.CFG_24KHZ)) == strip(so.layer_plan(so.CFG_24KHZ))


def test_golden_vectors():
    g = np.load(os.path.join(ROOT, "tests", "golden", "seanet_golden.npz"))
    for name, cfg in (("tiny", so.CFG_TINY), ("k24", so.CFG_24KHZ)):
        P = so.make_weights(cfg, int(g[f"{name}_seed"]))
        lat = so.encoder(g[f"{name}_wav"], P, cfg)
        assert rel(lat, g[f"{name}_lat"]) < 1e-5
        wav = so.decoder(g[f"{name}_lat"], P, cfg)
        assert rel(wav, g[f"{name}_out"]) < 1e-5


def test_random_state_dict_is_a_fresh_model():
    """`encodec_model_24khz(pretrained=False)` holds PyTorch-default-initialised tensors of the right shapes; g = |v| makes the folded
    weight equal v; a seed makes it reproducible."""
    import torch
    sd = codec.random_state_dict(codec.CFG_24KHZ, seed=3)
    assert {k: tuple(v.shape) for k, v in sd.items() if not k.startswith("quantizer")} == so.param_shapes(so.CFG_24KHZ)
    assert sum(k.startswith("quantizer.layers.") for k in sd) == 32 and tuple(sd["quantizer.layers.31.codebook.embed"].shape) == (1024, 128)
    k = "decoder.layers.3.conv.parametrizations.weight."
    v = sd[k + "original1"].numpy()
    assert np.abs(so.fold_weight_norm(sd[k + "original0"].numpy(), v) - v).max() < 1e-6
    assert float(sd[k + "original1"].abs().max()) <= 1 / np.sqrt(256 * 16) + 1e-7           # fan_in of ConvTranspose1d(512, 256, 16)
    again = codec.random_state_dict(codec.CFG_24KHZ, seed=3)
    assert all(torch.equal(sd[n], again[n]) for n in sd)


def test_algorithmic_flops_per_second_of_audio():
    """DESIGN.md 3.5 / bench.py's codec roofline: 2.98 GFLOP per second of audio for either stack of the 24 kHz model."""
    enc = codec.stack_flops(codec.CFG_24KHZ, "encoder", 24000)
    dec = codec.stack_flops(codec.CFG_24KHZ, "decoder", 75)
    assert abs(enc / 1e9 - 2.9795) < 1e-3 and abs(dec / 1e9 - 2.9795) < 1e-3
    # cross-check one layer by hand: the k = 16, stride 8 down-sampling convolution 256 -> 512 at 75 frames/s
    assert 2 * 256 * 512 * 16 * 75 == 314572800


def test_num_quantizers_and_key_dialects():
    assert so.num_quantizers(6.0) == 8 and so.num_quantizers(1.5) == 2 and so.num_quantizers(24.0) == 32
    nk = codec.normalise_key
    assert nk("encoder.model.3.conv.conv.weight_g") == "encoder.layers.3.conv.parametrizations.weight.original0"
    assert nk("encoder.model.1.block.1.conv.conv.weight_v") == "encoder.layers.1.block.1.conv.parametrizations.weight.original1"
    assert nk("encoder.model.1.shortcut.conv.conv.bias") == "encoder.layers.1.shortcut.conv.bias"
    assert nk("decoder.model.3.convtr.convtr.weight_g") == "decoder.layers.3.conv.parametrizations.weight.original0"
    assert nk("encoder.model.13.lstm.weight_ih_l0") == "encoder.layers.13.lstm.weight_ih_l0"
    assert nk("quantizer.vq.layers.7._codebook.embed") == "quantizer.layers.7.codebook.embed"
    assert nk("encoder.layers.0.conv.parametrizations.weight.original1") == "encoder.layers.0.conv.parametrizations.weight.original1"
    assert nk("decoder.layers.3.conv.weight_g") == "decoder.layers.3.conv.parametrizations.weight.original0"


# ------------------------------------------------------------------------------------------------ the C ABI
def test_header_symbols_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "prompt_tts_seanet.h")).read()
    declared = sorted(set(re.findall(r"\b(pt_sn_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(codec.EXPORTS)
    if not os.path.exists(codec.SEANET_LIB_PATH):
        pytest.skip("libpt_seanet.so not built")
    lib = C.CDLL(codec.SEANET_LIB_PATH)          # loading needs libcudart only; no compute call is made here
    for s in declared:
        assert hasattr(lib, s), s
    assert lib.pt_sn_version() == 1
    # ctypes mirror of pt_sn_conv_t: six pointers then eleven ints (padded to the pointer alignment)
    assert C.sizeof(codec.ConvDesc) == 6 * 8 + 12 * 4
    body = re.sub(r"/\*.*?\*/", "", re.search(r"typedef struct \{(.*?)\} pt_sn_conv_t;", hdr, re.S).group(1), flags=re.S)
    names = [n for n in re.findall(r"[A-Za-z_]\w*", body) if n not in ("const", "float", "int")]
    assert names == [f[0] for f in codec.ConvDesc._fields_]


def test_argument_validation_needs_no_gpu():
    """Every entry point validates before it touches the CUDA runtime: bad descriptors return -1 with a message (no launch is
    attempted, so this runs in the CPU tier)."""
    if not os.path.exists(codec.SEANET_LIB_PATH):
        pytest.skip("libpt_seanet.so not built")
    lib = codec.seanet_lib()
    buf = np.zeros(64, np.float32)
    p = buf.ctypes.data

    def conv(**kw):
        f = dict(x=p, w=p, bias=0, res=0, y=p, y_elu=0, B=1, Ci=1, Co=1, Lin=16, Lout=16, K=3, stride=1, dil=1, pad_left=2, reflect=1, Co_pad=8)
        f.update(kw)
        return codec.ConvDesc(**f)

    cases = [("conv1d", conv(y=0), "neither y nor y_elu"), ("conv1d", conv(x=0), "x and w must be set"), ("conv1d", conv(K=0), "bad sizes"),
             ("conv1d", conv(Lin=2, pad_left=2), "shorter than its reflect padding"),
             ("conv1d", conv(Lout=2**31 - 8, stride=8, reflect=0), "too long"),
             ("conv1d_packed", conv(Co=9, Co_pad=8), "Co_pad"), ("conv1d_packed", conv(Co_pad=12), "Co_pad"),
             ("conv_transpose1d", conv(dil=2), "dilation"), ("conv_transpose1d", conv(Lout=64, pad_left=0), "exceeds the full output length"),
             ("conv_transpose1d_packed", conv(Co_pad=4), "Co_pad")]
    for name, d, msg in cases:
        rc = getattr(lib, "pt_sn_" + name)(C.addressof(d), None)
        assert rc == -1 and msg in lib.pt_sn_last_error().decode(), (name, msg, rc, lib.pt_sn_last_error())
    assert lib.pt_sn_linear_rows(p, p, 0, p, 1, 3, 4, None) == -1 and b"multiples of 4" in lib.pt_sn_last_error()
    assert lib.pt_sn_linear_rows(p + 4, p, 0, p, 1, 4, 4, None) == -1 and b"aligned" in lib.pt_sn_last_error()
    assert lib.pt_sn_lstm_step(p, p, p, p, 0, 1, 6, None) == -1 and b"multiple of 4" in lib.pt_sn_last_error()
    assert lib.pt_sn_lstm_seq(p, p, p, p, 0, 1, 8, None) == -1
    assert lib.pt_sn_pack_conv_weight(p, p, 9, 1, 1, 8, 0, None) == -1
    assert lib.pt_sn_weight_norm_fold(p, p, p, 0, 4, None) == -1
    assert lib.pt_sn_launch_count() == 0


def test_product_raises_without_gpu():
    """Run with no CUDA device visible (CUDA_VISIBLE_DEVICES empty), so that a machine with a GPU checks it too."""
    code = r'''
import sys
sys.path.insert(0, %r)
import pytest
from prompt_tts_b200 import codec
from prompt_tts_b200._lib import PtError
with pytest.raises(PtError):
    codec.EncodecModel()
with pytest.raises(PtError):
    codec.EncodecModel.encodec_model_24khz(pretrained=False)
print("OK")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


# ------------------------------------------------------------------------------------------------ kernel bodies vs oracle
CONV_CASES = [
    # B, Ci, Co, L, K, stride, dil, causal, reflect
    (2, 1, 4, 700, 7, 1, 1, True, True),
    (1, 3, 13, 1100, 7, 1, 1, False, True),
    (2, 8, 16, 523, 4, 2, 1, True, True),
    (1, 5, 9, 601, 8, 4, 1, True, True),
    (1, 4, 8, 333, 10, 5, 1, False, True),
    (2, 6, 12, 129, 16, 8, 1, True, True),
    (1, 6, 3, 97, 3, 1, 2, True, True),
    (1, 6, 3, 97, 3, 1, 4, False, False),
    (2, 7, 1, 50, 1, 1, 1, True, True),
    (1, 2, 5, 41, 5, 3, 1, True, False),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv1d_body_matches_oracle(drv, case):
    B, Ci, Co, L, K, stride, dil, causal, reflect = case
    rng = np.random.default_rng(hash(case) % 2**32)
    x = rng.standard_normal((B, Ci, L)).astype(np.float32)
    w = rng.standard_normal((Co, Ci, K)).astype(np.float32) / np.float32(np.sqrt(Ci * K))
    b = rng.standard_normal(Co).astype(np.float32)
    ref = so.conv1d(x, w, b, stride, dil, causal, "reflect" if reflect else "constant")
    Lout = ref.shape[-1]
    res = rng.standard_normal(ref.shape).astype(np.float32)
    y, ye = drv.empty(B, Co, Lout), drv.empty(B, Co, Lout)
    left, _ = so.pad_amounts(K, stride, dil, causal)
    d = codec.ConvDesc(x.ctypes.data, w.ctypes.data, b.ctypes.data, res.ctypes.data, y.ctypes.data, ye.ctypes.data,
                       B, Ci, Co, L, Lout, K, stride, dil, left, 1 if reflect else 0)
    drv.call("conv1d", C.addressof(d))
    assert rel(y, ref + res) < 2e-6
    assert rel(ye, so.elu(ref + res)) < 2e-6
    # no residual, no bias, only the activated copy
    ye2 = drv.empty(B, Co, Lout)
    d = codec.ConvDesc(x.ctypes.data, w.ctypes.data, 0, 0, 0, ye2.ctypes.data, B, Ci, Co, L, Lout, K, stride, dil, left, 1 if reflect else 0)
    drv.call("conv1d", C.addressof(d))
    assert rel(ye2, so.elu(ref - b[None, :, None])) < 2e-6
    # packed weights (8 or 16 output channels per thread, interior / boundary loops)
    for cop in sorted({codec.SeanetStack.co_pad(Co), -(-Co // 8) * 8}):
        wp = drv.empty(Ci, K, cop)
        drv.call("pack_conv_weight", w.ctypes.data, wp.ctypes.data, Co, Ci, K, cop, 0)
        assert np.array_equal(wp[:, :, :Co], w.transpose(1, 2, 0)) and not wp[:, :, Co:].any()
        y3, ye3 = drv.empty(B, Co, Lout), drv.empty(B, Co, Lout)
        d = codec.ConvDesc(x.ctypes.data, wp.ctypes.data, b.ctypes.data, res.ctypes.data, y3.ctypes.data, ye3.ctypes.data,
                           B, Ci, Co, L, Lout, K, stride, dil, left, 1 if reflect else 0, cop)
        drv.call("conv1d_packed", C.addressof(d))
        assert np.array_equal(y3, y), cop               # same products in the same order as the reference-layout kernel
        assert np.array_equal(ye3, ye)


CONVTR_CASES = [
    # B, Ci, Co, L, K, stride, causal
    (2, 8, 4, 75, 16, 8, True),
    (1, 6, 5, 130, 10, 5, True),
    (1, 4, 3, 300, 8, 4, False),
    (2, 4, 2, 700, 4, 2, True),
    (1, 3, 7, 40, 7, 3, True),
    (1, 3, 2, 40, 5, 1, False),
    (1, 5, 1, 20, 6, 6, True),
]


@pytest.mark.parametrize("case", CONVTR_CASES)
def test_conv_transpose_body_matches_oracle(drv, case):
    B, Ci, Co, L, K, stride, causal = case
    rng = np.random.default_rng(hash(case) % 2**32)
    x = rng.standard_normal((B, Ci, L)).astype(np.float32)
    w = rng.standard_normal((Ci, Co, K)).astype(np.float32) / np.float32(np.sqrt(Ci * 2))
    b = rng.standard_normal(Co).astype(np.float32)
    ref = so.conv_transpose1d(x, w, b, stride, causal)
    assert ref.shape[-1] == L * stride
    total = K - stride
    left = 0 if causal else total - total // 2
    y, ye = drv.empty(*ref.shape), drv.empty(*ref.shape)
    d = codec.ConvDesc(x.ctypes.data, w.ctypes.data, b.ctypes.data, 0, y.ctypes.data, ye.ctypes.data,
                       B, Ci, Co, L, ref.shape[-1], K, stride, 1, left, 0)
    drv.call("conv_transpose1d", C.addressof(d))
    assert rel(y, ref) < 2e-6
    assert rel(ye, so.elu(ref)) < 2e-6
    cop = codec.SeanetStack.co_pad(Co)
    wp = drv.empty(Ci, K, cop)
    drv.call("pack_conv_weight", w.ctypes.data, wp.ctypes.data, Co, Ci, K, cop, 1)
    assert np.array_equal(wp[:, :, :Co], w.transpose(0, 2, 1)) and not wp[:, :, Co:].any()
    y3, ye3 = drv.empty(*ref.shape), drv.empty(*ref.shape)
    d = codec.ConvDesc(x.ctypes.data, wp.ctypes.data, b.ctypes.data, 0, y3.ctypes.data, ye3.ctypes.data,
                       B, Ci, Co, L, ref.shape[-1], K, stride, 1, left, 0, cop)
    drv.call("conv_transpose1d_packed", C.addressof(d))
    assert np.array_equal(y3, y) and np.array_equal(ye3, ye)


def test_weight_norm_and_lstm_packing(drv):
    rng = np.random.default_rng(0)
    for shape in ((5, 3, 7), (130, 2, 1), (4, 6, 16)):
        v = rng.standard_normal(shape).astype(np.float32)
        g = rng.uniform(0.5, 2.0, (shape[0], 1, 1)).astype(np.float32)
        w = drv.empty(*shape)
        drv.call("weight_norm_fold", v.ctypes.data, g.ctypes.data, w.ctypes.data, shape[0], shape[1] * shape[2])
        assert rel(w, so.fold_weight_norm(g, v)) < 1e-6
    H = 12
    W = rng.standard_normal((4 * H, H)).astype(np.float32)
    t4 = drv.empty(H, H, 4)
    drv.call("lstm_pack", W.ctypes.data, t4.ctypes.data, H)
    assert np.array_equal(t4, W.reshape(4, H, H).transpose(2, 1, 0))          # [k][j][q] = W[q*H + j][k]
    bi, bh = rng.standard_normal(4 * H).astype(np.float32), rng.standard_normal(4 * H).astype(np.float32)
    b4 = drv.empty(H, 4)
    drv.call("lstm_pack_bias", bi.ctypes.data, bh.ctypes.data, b4.ctypes.data, H)
    assert np.array_equal(b4, (bi + bh).reshape(4, H).T)


def test_transposes_and_linear_rows(drv):
    rng = np.random.default_rng(1)
    B, Cn, T = 3, 20, 37
    x = rng.standard_normal((B, Cn, T)).astype(np.float32)
    out = drv.empty(T, B, Cn)
    drv.call("ncl_to_tbc", x.ctypes.data, out.ctypes.data, B, Cn, T)
    assert np.array_equal(out, x.transpose(2, 0, 1))
    h = rng.standard_normal((T, B, Cn)).astype(np.float32)
    y, ye = drv.empty(B, Cn, T), drv.empty(B, Cn, T)
    drv.call("tbc_add_to_ncl", h.ctypes.data, x.ctypes.data, y.ctypes.data, ye.ctypes.data, B, Cn, T)
    assert np.array_equal(y, h.transpose(1, 2, 0) + x)
    assert rel(ye, so.elu(h.transpose(1, 2, 0) + x)) < 1e-6
    for R, Kd, N in ((7, 20, 80), (130, 64, 256), (1, 4, 4), (9, 512, 2048)):
        a = rng.standard_normal((R, Kd)).astype(np.float32)
        wt = rng.standard_normal((Kd, N)).astype(np.float32)
        bias = rng.standard_normal(N).astype(np.float32)
        o = drv.empty(R, N)
        drv.call("linear_rows", a.ctypes.data, wt.ctypes.data, bias.ctypes.data, o.ctypes.data, R, Kd, N)
        assert rel(o, a.astype(np.float64) @ wt.astype(np.float64) + bias) < 2e-6


@pytest.mark.parametrize("B,H,T", [(1, 16, 9), (3, 64, 21), (5, 132, 6), (37, 32, 5)])
def test_lstm_sequencing_matches_oracle(drv, B, H, T):
    cfg = dict(so.CFG_TINY, num_filters=H // 16)
    rng = np.random.default_rng(B * 100 + H)
    P = {}
    prefix = "encoder.layers.13"
    for l in range(2):
        for n, shape in (("weight_ih", (4 * H, H)), ("weight_hh", (4 * H, H)), ("bias_ih", (4 * H,)), ("bias_hh", (4 * H,))):
            P[f"{prefix}.lstm.{n}_l{l}"] = (rng.uniform(-1, 1, shape) / np.sqrt(H) * 2).astype(np.float32)
    x = rng.standard_normal((B, H, T)).astype(np.float32)
    ref = so.lstm(x, P, prefix, 2)
    st = codec.SeanetStack(cfg, "encoder", drv)
    for l in range(2):
        for n in ("weight_ih", "weight_hh"):
            t4 = drv.empty(H, H, 4)
            drv.call("lstm_pack", P[f"{prefix}.lstm.{n}_l{l}"].ctypes.data, t4.ctypes.data, H)
            st.w[f"{prefix}.{n}_l{l}"] = t4
        b4 = drv.empty(H, 4)
        drv.call("lstm_pack_bias", P[f"{prefix}.lstm.bias_ih_l{l}"].ctypes.data, P[f"{prefix}.lstm.bias_hh_l{l}"].ctypes.data, b4.ctypes.data, H)
        st.w[f"{prefix}.bias_l{l}"] = b4
    outs = {}
    for fast in (False, True):
        st.lstm_whole = fast
        drv.calls.clear()
        y, ye = st._lstm(prefix, x, B, H, T, True, True)
        assert rel(y, ref) < 5e-6
        assert rel(ye, so.elu(ref)) < 5e-6
        assert drv.calls.count("lstm_seq") == (2 if fast else 0) and drv.calls.count("lstm_step") == (0 if fast else 2 * T)
        outs[fast] = y
    assert np.array_equal(outs[True], outs[False])      # the whole-sequence kernel does the step kernel's arithmetic


# ------------------------------------------------------------------------------------------------ whole stacks through the product's sequencing
@pytest.mark.parametrize("fast", [True, False])
@pytest.mark.parametrize("name,S,B", [("tiny", 3203, 2), ("tiny_noshortcut", 2900, 1), ("tiny_noncausal", 3333, 1), ("tiny_res2_zero", 3200, 1),
                                      ("k24", 2881, 1)])
def test_stacks_match_oracle(drv, name, S, B, fast):
    cfg = {"tiny": so.CFG_TINY, "k24": so.CFG_24KHZ, "tiny_noshortcut": dict(so.CFG_TINY, use_conv_shortcut=False),
           "tiny_noncausal": dict(so.CFG_TINY, use_causal_conv=False),
           "tiny_res2_zero": dict(so.CFG_TINY, num_residual_layers=2, dilation_growth_rate=3, pad_mode="constant")}[name]
    P = so.make_weights(cfg, 11)
    x = (np.random.default_rng(2).standard_normal((B, 1, S)) * 0.3).astype(np.float32)
    if name == "k24" and not fast:
        pytest.skip("the 24 kHz widths run once, on the default path (CPU time)")
    enc = codec.SeanetStack(cfg, "encoder", drv, fast=fast)
    enc.prepare({k: drv.upload(P[k]) for k in enc.param_names()})
    drv.calls.clear()
    lat, T = enc.forward(x, B, S)
    assert ("conv1d_packed" in drv.calls) == fast and ("conv1d" in drv.calls) == (not fast)
    lat_ref = so.encoder(x, P, cfg)
    assert lat.shape == lat_ref.shape and T == lat_ref.shape[-1]
    assert rel(lat, lat_ref) < 2e-5
    dec = codec.SeanetStack(cfg, "decoder", drv, fast=fast)
    dec.prepare({k: drv.upload(P[k]) for k in dec.param_names()})
    wav, L = dec.forward(lat_ref, B, T)
    wav_ref = so.decoder(lat_ref, P, cfg)
    assert wav.shape == wav_ref.shape and L == 320 * T
    assert rel(wav, wav_ref) < 2e-5
    assert not np.isnan(wav).any() and not np.isnan(lat).any()


# ------------------------------------------------------------------------------------------------ randomised shapes
def _rand_conv_case(rng):
    K = int(rng.integers(1, 9))
    stride = int(rng.integers(1, K + 1))
    dil = int(rng.integers(1, 4)) if stride == 1 else 1
    reach = (K - 1) * dil + 1
    L = int(rng.integers(reach + stride + 1, 700))
    return dict(B=int(rng.integers(1, 3)), Ci=int(rng.integers(1, 7)), Co=int(rng.integers(1, 20)), L=L, K=K, stride=stride, dil=dil,
                causal=bool(rng.integers(0, 2)), reflect=bool(rng.integers(0, 2)))


@pytest.mark.parametrize("seed", range(24))
def test_conv_bodies_random_shapes(drv, seed):
    """Ragged sizes the fixed cases do not hit: channel counts around the 8 / 16 tile edges, lengths around the 512-sample block
    tile, strides that do not divide the kernel, dilation with and without reflection."""
    rng = np.random.default_rng(1000 + seed)
    c = _rand_conv_case(rng)
    B, Ci, Co, L, K, stride, dil = c["B"], c["Ci"], c["Co"], c["L"], c["K"], c["stride"], c["dil"]
    x = rng.standard_normal((B, Ci, L)).astype(np.float32)
    w = rng.standard_normal((Co, Ci, K)).astype(np.float32)
    b = rng.standard_normal(Co).astype(np.float32)
    try:
        ref = so.conv1d(x, w, b, stride, dil, c["causal"], "reflect" if c["reflect"] else "constant")
    except ValueError:
        pytest.skip("input shorter than its reflect padding")
    left, _ = so.pad_amounts(K, stride, dil, c["causal"])
    Lout = ref.shape[-1]
    for cop, name in ((0, "conv1d"), (codec.SeanetStack.co_pad(Co), "conv1d_packed"), (-(-Co // 8) * 8, "conv1d_packed")):
        wk = w
        if cop:
            wk = drv.empty(Ci, K, cop)
            drv.call("pack_conv_weight", w.ctypes.data, wk.ctypes.data, Co, Ci, K, cop, 0)
        y = drv.empty(B, Co, Lout)
        d = codec.ConvDesc(x.ctypes.data, wk.ctypes.data, b.ctypes.data, 0, y.ctypes.data, 0, B, Ci, Co, L, Lout, K, stride, dil, left,
                           1 if c["reflect"] else 0, cop)
        drv.call(name, C.addressof(d))
        assert rel(y, ref) < 3e-6, (c, name, cop)
    # transposed: the same (K, stride) family, all of K - stride trimmed at the end (causal) or split (non-causal)
    wt = rng.standard_normal((Ci, Co, K)).astype(np.float32)
    Lt = int(rng.integers(1, 200))
    xt = rng.standard_normal((B, Ci, Lt)).astype(np.float32)
    reft = so.conv_transpose1d(xt, wt, b, stride, c["causal"])
    total = K - stride
    tl = 0 if c["causal"] else total - total // 2
    for cop, name in ((0, "conv_transpose1d"), (codec.SeanetStack.co_pad(Co), "conv_transpose1d_packed")):
        wk = wt
        if cop:
            wk = drv.empty(Ci, K, cop)
            drv.call("pack_conv_weight", wt.ctypes.data, wk.ctypes.data, Co, Ci, K, cop, 1)
        y = drv.empty(*reft.shape)
        d = codec.ConvDesc(xt.ctypes.data, wk.ctypes.data, b.ctypes.data, 0, y.ctypes.data, 0, B, Ci, Co, Lt, reft.shape[-1], K, stride, 1, tl, 0, cop)
        drv.call(name, C.addressof(d))
        assert rel(y, reft) < 3e-6, (c, name, cop)


@pytest.mark.parametrize("seed", range(6))
def test_lstm_bodies_random_shapes(drv, seed):
    """Whole-sequence body == step body bit for bit, for batch sizes around the 32-sequence chunk and widths around the block tile."""
    rng = np.random.default_rng(2000 + seed)
    B, H, T = int(rng.integers(1, 70)), 4 * int(rng.integers(1, 40)), int(rng.integers(1, 6))
    xg = rng.standard_normal((T, B, H, 4)).astype(np.float32)
    whh = (rng.standard_normal((H, H, 4)) / np.sqrt(H)).astype(np.float32)
    out = []
    for whole in (True, False):
        hseq, c = drv.empty(T, B, H), drv.empty(B, H)
        if whole:
            drv.call("lstm_seq", xg.ctypes.data, whh.ctypes.data, hseq.ctypes.data, c.ctypes.data, T, B, H)
        else:
            for t in range(T):
                drv.call("lstm_step", xg.ctypes.data, whh.ctypes.data, hseq.ctypes.data, c.ctypes.data, t, B, H)
        assert not np.isnan(hseq).any() and not np.isnan(c).any()
        out.append((hseq, c))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    # and against a plain numpy recurrence on the packed operands: gates = xg[t] + h @ W, order i, f, g, o
    h, cc = np.zeros((B, H), np.float32), np.zeros((B, H), np.float32)
    sig = lambda a: 1.0 / (1.0 + np.exp(-a))
    for t in range(T):
        g = xg[t].astype(np.float64) + np.einsum("bk,kjq->bjq", h.astype(np.float64), whh.astype(np.float64))
        cc = sig(g[..., 1]) * cc + sig(g[..., 0]) * np.tanh(g[..., 2])
        h = sig(g[..., 3]) * np.tanh(cc)
        assert rel(out[0][0][t], h) < 1e-5


def test_encodec_dialect_round_trip_for_every_tensor():
    """Every tensor name of the 24 kHz model, written the way encodec 0.1.1 names it (`model.N`, `conv.conv` / `convtr.convtr`,
    `weight_g` / `weight_v`, `vq.layers.N._codebook`), maps back onto the name this package stores."""
    plan = codec.layer_plan(codec.CFG_24KHZ)
    transposed = {f"{side}.layers.{i}" for side, p in plan.items() for i, kind, _ in p if kind == "convtr"}
    names = list(so.param_shapes(so.CFG_24KHZ)) + [f"quantizer.layers.{q}.codebook.embed" for q in range(32)]
    for n in names:
        old = n
        if n.startswith(("encoder.", "decoder.")):
            old = n.replace(".layers.", ".model.", 1)
            inner = "convtr.convtr" if n.split(".conv.")[0] in transposed else "conv.conv"
            old = old.replace(".conv.parametrizations.weight.original0", f".{inner}.weight_g").replace(
                ".conv.parametrizations.weight.original1", f".{inner}.weight_v").replace(".conv.bias", f".{inner}.bias")
        else:
            old = n.replace("quantizer.layers.", "quantizer.vq.layers.").replace(".codebook.embed", "._codebook.embed")
        assert old != n and codec.normalise_key(old) == n, (n, old, codec.normalise_key(old))
