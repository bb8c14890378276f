"""ctypes binding of libpt_b200.so (include/prompt_tts_b200.h).

There is no fallback: if the shared library is missing or a call returns non-zero this raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PT_B200_LIB") or os.path.join(_HERE, "libpt_b200.so")   # the override is for A/B runs of two builds


class Operand(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("dim", C.c_int64 * 4), ("stride", C.c_int64 * 4),
                ("kmajor", C.c_int32), ("batched", C.c_int32)]


class Segment(C.Structure):
    _fields_ = [("a_idx", C.c_int32), ("b_idx", C.c_int32), ("a_k0", C.c_int32), ("b_k0", C.c_int32),
                ("a_mn_shift", C.c_int32), ("b_mn_shift", C.c_int32), ("nk", C.c_int32), ("nrep", C.c_int32),
                ("rep_is_batch", C.c_int32), ("rep_c2_0", C.c_int32), ("b_k0_z2", C.c_int32)]


class Gemm(C.Structure):
    _fields_ = [("a", Operand * 2), ("b", Operand * 2), ("seg", Segment * 8), ("nseg", C.c_int32),
                ("M", C.c_int32), ("N", C.c_int32), ("nz2", C.c_int32), ("nz3", C.c_int32),
                ("splitk", C.c_int32), ("block_n", C.c_int32),
                ("out", C.c_void_p), ("out_dtype", C.c_int32),
                ("out_stride_m", C.c_int64), ("out_stride_z2", C.c_int64), ("out_stride_z3", C.c_int64),
                ("alpha", C.c_float), ("bias", C.c_void_p), ("bias_z2", C.c_void_p), ("residual", C.c_void_p),
                ("res_stride_m", C.c_int64), ("res_stride_z2", C.c_int64), ("res_stride_z3", C.c_int64),
                ("bias_z2_stride", C.c_int64), ("out_stride_n", C.c_int64), ("out_transposed", C.c_int32)]


class Attn(C.Structure):
    _fields_ = [("q", C.c_void_p), ("q_rs", C.c_int64), ("q_bs", C.c_int64),
                ("k", C.c_void_p), ("v", C.c_void_p), ("kv_rs", C.c_int64), ("kv_bs", C.c_int64),
                ("o", C.c_void_p), ("o_rs", C.c_int64), ("o_bs", C.c_int64),
                ("lse", C.c_void_p),
                ("d_o", C.c_void_p), ("do_rs", C.c_int64), ("do_bs", C.c_int64),
                ("dq", C.c_void_p), ("dq_rs", C.c_int64), ("dq_bs", C.c_int64),
                ("dk", C.c_void_p), ("dv", C.c_void_p), ("dkv_rs", C.c_int64), ("dkv_bs", C.c_int64),
                ("delta", C.c_void_p),
                ("B", C.c_int32), ("H", C.c_int32), ("Lq", C.c_int32), ("Lk", C.c_int32), ("d", C.c_int32),
                ("scale", C.c_float)]


OUT_BF16, OUT_F32, OUT_F32_ATOMIC_ADD = 0, 1, 2

_lib = None


class PtError(RuntimeError):
    pass


def lib():
    """Load the CUDA library; raise (never fall back) when it is not there."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PtError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU / PyTorch fallback for the hot path)")
        _lib = C.CDLL(LIB_PATH)
        _lib.pt_last_error.restype = C.c_char_p
        _lib.pt_version.restype = C.c_int
        _lib.pt_launch_count.restype = C.c_ulonglong
        _lib.pt_rvq_encode_tc_scratch_bytes.restype = C.c_size_t
        _lib.pt_rvq_encode_tc_scratch_bytes.argtypes = [C.c_int, C.c_int]
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise PtError(f"{what}: rc={rc}: {lib().pt_last_error().decode()}")


def call(name: str, *args) -> None:
    """Call `pt_<name>` with ctypes-converted args and raise on a non-zero return."""
    fn = getattr(lib(), "pt_" + name)
    check(fn(*args), "pt_" + name)


# ---------------------------------------------------------------------------------------------
# argtypes for every entry point of include/prompt_tts_b200.h  (p = pointer, i = int, l = int64, f = float)
# ---------------------------------------------------------------------------------------------
_SIGS = {
    "check_device": "i",
    "set_sm_reserve": "i",
    "gemm": "pp",
    "attn_fwd": "pp",
    "attn_bwd": "pp",
    "groupnorm_stats": "ppiiiifp",
    "groupnorm_apply": "pppppiiiiip",
    "groupnorm_fwd": "pppppiiiifip",
    "groupnorm_bwd": "ppppppppppiiiiip",
    "layernorm_fwd": "ppppplifp",
    "layernorm_bwd": "pppppppplip",
    "softmax_fwd": "pplillp",
    "softmax_bwd": "ppplillfp",
    "geglu_fwd": "pplip",
    "geglu_bwd": "ppplip",
    "add_bf16": "ppplp",
    "silu_f32_to_bf16": "pplp",
    "silu_bwd_f32": "ppplp",
    "copy2d_bf16": "plpllip",
    "upsample2_fwd": "ppiiip",
    "upsample2_bwd": "ppiiip",
    "ncl_f32_to_nlc_bf16": "ppiiip",
    "nlc_bf16_to_ncl_f32": "ppiiip",
    "cast_f32_to_bf16": "pplp",
    "cast_bf16_to_f32": "pplp",
    "pack_conv_weight": "ppiiip",
    "unpack_conv_wgrad": "ppiiiip",
    "colsum_bf16": "plplip",
    "colsum_bf16_lite": "plplip",
    "batch_colsum_bf16": "ppliiip",
    "conv_in_fwd": "ppppiiiip",
    "conv_in_bwd": "ppppiiiip",
    "conv_out_fwd": "ppppiiiip",
    "conv_out_bwd": "ppppppiiiip",
    "time_sinusoid": "ppiip",
    "text_embed_fwd": "ppppiiiip",
    "text_embed_bwd": "pppiiiip",
    "add_noise": "ppppppilp",
    "mse_fwd_bwd": "pppplfp",
    "diffusion_loss": "ppppppppiliffp",
    "ddpm_step": "pppppliiffp",
    "ddim_step": "ppppppliifffffp",
    "dpmpp_step": "pppppppliifffiffp",
    "ddpm_step_pred": "pppppliiffip",
    "ddim_step_pred": "ppppppliifffffip",
    "dpmpp_step_pred": "pppppppliifffiffip",
    "cond_select_bf16": "pppilp",
    "cfg_combine": "pplfp",
    "rows_add_bias_bf16": "ppplip",
    "rvq_encode_ws": "ppppiiiiip",
    "rvq_cb_sq": "ppiiip",
    "rvq_encode_tc": "pppipiiiiip",
    "rvq_tc_debug_scores": "p",
    "rvq_decode": "pppiiiiip",
    "rvq_decode_ws": "ppppiiiiip",
    "codes_affine": "pplp",
    "codes_affine_inv": "pplp",
    "sumsq_f32": "plpp",
    "adamw_step": "pppplfffffipffp",
    "sumsq_bf16": "plpp",
    "adamw_prepare": "ppp",
    "sumsq_partials": "pilpip",
    "adamw_prepare_det": "ppip",
    "adamw_step_dev": "ppippplpp",
    "ema_prepare": "pp",
    "adamw_ema_step_dev": "ppipppplppp",
    "ema_swap": "ppplp",
}
_CT = {"p": C.c_void_p, "i": C.c_int, "l": C.c_int64, "f": C.c_float}
EXPORTS = ["pt_version", "pt_last_error", "pt_launch_count", "pt_gemm_last_tile", "pt_rvq_encode_tc_scratch_bytes"] + ["pt_" + k for k in _SIGS]


def _bind(l):
    for name, sig in _SIGS.items():
        fn = getattr(l, "pt_" + name)
        fn.argtypes = [_CT[c] for c in sig]
        fn.restype = C.c_int


_orig_lib = lib


def lib():  # noqa: F811  (wraps the loader above with argtype binding)
    global _lib
    first = _lib is None
    l = _orig_lib()
    if first:
        _bind(l)
    return l
