"""Build + ctypes binding of ``libw2s_b200.so`` (C ABI declared in ``include/w2s_b200.h``).

The shared library is compiled in-tree with ``nvcc`` for sm_100a only.  There is no CPU fallback: if the
library cannot be loaded every compute entry point raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
REPO_DIR = PKG_DIR.parent
# W2S_LIB_VARIANT=name selects libw2s_b200_<name>.so (A/B builds with other W2S_NVCC_FLAGS, tools/ab_build.sh)
LIB_PATH = PKG_DIR / ("libw2s_b200" + ("_" + os.environ["W2S_LIB_VARIANT"] if os.environ.get("W2S_LIB_VARIANT") else "") + ".so")
SOURCES = [PKG_DIR / "csrc" / "capi.cu"]
HEADERS = sorted((PKG_DIR / "csrc").glob("*.cuh")) + [REPO_DIR / "include" / "w2s_b200.h"]

MAX_BLOCKS = 12
MAX_MIXER_LAYERS = 8
MAX_SIGNALS = 4
MAX_SEQ_BLOCKS = 4
MAX_DILATIONS = 8
STREAM_MAX_LAYERS = 32
STREAM_MAX_DILATIONS = 16
STREAM_MAX_KERNEL = 16
STREAM_MAX_FEATURES = 256
ABI_VERSION = 11

PRO_NONE, PRO_NORM, PRO_NORM_RES, PRO_FIR, PRO_NORM_RES_X, PRO_DNORM = 0, 1, 2, 3, 4, 5
EPI_STATS, EPI_BIAS_GELU, EPI_LN_GELU, EPI_LN_GELU_RES, EPI_PLAIN, EPI_ACT_BWD = 0, 1, 2, 3, 4, 5


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; cannot build libw2s_b200.so")
    return p


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
    if not force and LIB_PATH.exists():
        newest = max(p.stat().st_mtime for p in SOURCES + HEADERS)
        if LIB_PATH.stat().st_mtime >= newest:
            return LIB_PATH
    cmd = [
        nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
        "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "1886", "-o", str(LIB_PATH),
    ] + [str(s) for s in SOURCES]
    cmd[1:1] = os.environ.get("W2S_NVCC_FLAGS", "").split()  # e.g. -DW2S_DEBUG_KNOCKOUTS for tools/dbg_flags.sh
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{res.stdout}\n{res.stderr}")
    if verbose:
        print(res.stderr)
    return LIB_PATH


class PackJob(C.Structure):
    _fields_ = [("w", C.c_void_p), ("out", C.c_void_p), ("kind", C.c_int32), ("cout", C.c_int32), ("cin", C.c_int32),
                ("taps", C.c_int32), ("sn", C.c_int64), ("sc", C.c_int64), ("st", C.c_int64), ("split", C.c_int32),
                ("reserved", C.c_int32)]


class ConvCall(C.Structure):
    _fields_ = [
        ("cin", C.c_int32), ("cout", C.c_int32), ("taps", C.c_int32), ("stride", C.c_int32),
        ("dilation", C.c_int32), ("pad", C.c_int32),
        ("prologue", C.c_int32), ("epilogue", C.c_int32), ("has_ds", C.c_int32),
        ("B", C.c_int32), ("L_in", C.c_int32), ("L_out", C.c_int32),
        ("in_", C.c_void_p), ("in_res", C.c_void_p), ("in_stats", C.c_void_p),
        ("w", C.c_void_p), ("w_ds", C.c_void_p),
        ("out", C.c_void_p), ("out_ds", C.c_void_p), ("out_stats", C.c_void_p),
        ("row_mask", C.c_void_p), ("bias", C.c_void_p), ("ln_w", C.c_void_p), ("ln_b", C.c_void_p),
        ("res", C.c_void_p), ("head_w", C.c_void_p), ("head_b", C.c_void_p), ("logits", C.c_void_p),
        ("n_classes", C.c_int32), ("in_eps", C.c_float), ("ln_eps", C.c_float),
        ("out_stride", C.c_int32), ("out_offset", C.c_int32), ("out_rows", C.c_int32),
        ("x_raw", C.c_void_p), ("w_first", C.c_void_p), ("w_first_ds", C.c_void_p), ("T_raw", C.c_int32),
        ("in_wide", C.c_int32), ("out_wide", C.c_int32), ("force_split", C.c_int32),
        ("act_y", C.c_void_p), ("act_r", C.c_void_p), ("act_stats", C.c_void_p), ("act_a", C.c_void_p),
        ("act_dr", C.c_void_p), ("act_eps", C.c_float),
        ("dn_sums", C.c_void_p), ("dn_out", C.c_void_p), ("dn_upsample", C.c_int32),
    ]


class EncoderDesc(C.Structure):
    _fields_ = [
        ("n_blocks", C.c_int32), ("channels", C.c_int32 * MAX_BLOCKS), ("feature_dim", C.c_int32),
        ("norm_eps", C.c_float),
        ("w_first", C.c_void_p), ("w_first_ds", C.c_void_p),
        ("w_conv", (C.c_void_p * 3) * MAX_BLOCKS), ("w_ds", C.c_void_p * MAX_BLOCKS),
        ("w_lin", C.c_void_p), ("b_lin", C.c_void_p),
        ("wide_blocks", C.c_int32),
    ]


class MixerLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "in_w", "out_w", "ff1_w", "ff2_w", "in_b", "out_b", "ff1_b", "ff2_b", "ln1_w", "ln1_b", "ln2_w", "ln2_b")]


class MixerDesc(C.Structure):
    _fields_ = [
        ("n_layers", C.c_int32), ("feature_dim", C.c_int32), ("n_heads", C.c_int32), ("dim_ff", C.c_int32),
        ("ln_eps", C.c_float), ("cls", C.c_void_p), ("layer", MixerLayer * MAX_MIXER_LAYERS),
    ]


class SeqDesc(C.Structure):
    _fields_ = [
        ("n_blocks", C.c_int32), ("n_dilations", C.c_int32), ("kernel_size", C.c_int32),
        ("feature_dim", C.c_int32), ("n_classes", C.c_int32), ("ln_eps", C.c_float),
        ("w", (C.c_void_p * MAX_DILATIONS) * MAX_SEQ_BLOCKS),
        ("ln_w", (C.c_void_p * MAX_DILATIONS) * MAX_SEQ_BLOCKS),
        ("ln_b", (C.c_void_p * MAX_DILATIONS) * MAX_SEQ_BLOCKS),
        ("head_w", C.c_void_p), ("head_b", C.c_void_p),
    ]


class SeqStreamLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("w", "bias", "norm_w", "norm_b", "running_mean", "running_var")]


class SeqStreamDesc(C.Structure):
    _fields_ = [
        ("n_blocks", C.c_int32), ("n_dilations", C.c_int32), ("kernel_size", C.c_int32), ("feature_dim", C.c_int32),
        ("n_classes", C.c_int32), ("norm", C.c_int32), ("act", C.c_int32), ("eps", C.c_float),
        ("layer", SeqStreamLayer * STREAM_MAX_LAYERS), ("head_w", C.c_void_p), ("head_b", C.c_void_p), ("ring", C.c_void_p),
    ]


# name -> (restype, argtypes); every symbol declared in include/w2s_b200.h
SYMBOLS = {
    "w2s_abi_version": (C.c_int, []),
    "w2s_last_error": (C.c_char_p, []),
    "w2s_pack_conv_weight": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p]),
    "w2s_packed_conv_weight_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "w2s_conv_uses_split": (C.c_int, [C.c_int, C.c_int]),
    "w2s_encoder_conv_split": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "w2s_pack_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "w2s_pack_linear_frag": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "w2s_conv1d_fwd": (C.c_int, [C.POINTER(ConvCall), C.c_void_p]),
    "w2s_conv1d_fwd_pair": (C.c_int, [C.POINTER(ConvCall), C.POINTER(ConvCall), C.c_void_p]),
    "w2s_set_conv_impl": (C.c_int, [C.c_int]),
    "w2s_encoder_workspace_bytes": (C.c_size_t, [C.POINTER(EncoderDesc), C.c_int, C.c_int64, C.c_int]),
    "w2s_encoder_layout": (C.c_int, [C.POINTER(EncoderDesc), C.c_int, C.c_int64, C.POINTER(C.c_int64)]),
    "w2s_encoder_fwd": (C.c_int, [C.POINTER(EncoderDesc), C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_size_t,
                                  C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_encoder_fwd_pair": (C.c_int, [C.POINTER(EncoderDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.POINTER(EncoderDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_int64, C.c_size_t, C.c_int, C.c_void_p]),
    "w2s_epoch_mixer_fwd": (C.c_int, [C.POINTER(MixerDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                      C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "w2s_seqmixer_workspace_bytes": (C.c_size_t, [C.POINTER(SeqDesc), C.c_int, C.c_int, C.c_int]),
    "w2s_seqmixer_head_fwd": (C.c_int, [C.POINTER(SeqDesc), C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                        C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_argmax": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "w2s_gemm_tn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                              C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_longlong, C.c_float, C.c_void_p,
                              C.c_void_p]),
    "w2s_enc_act_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_enc_act_bwd": (C.c_int, [C.c_void_p] * 9 + [C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_enc_norm_bwd": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_first_conv_wgrad": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_first_conv_dgrad": (C.c_int, [C.c_void_p] * 7 + [C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_row_ln_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_longlong, C.c_int, C.c_float, C.c_void_p]),
    "w2s_row_ln_bwd": (C.c_int, [C.c_void_p] * 10 + [C.c_longlong, C.c_int, C.c_float, C.c_float, C.c_void_p]),
    "w2s_gelu_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "w2s_gelu_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "w2s_colsum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong,
                             C.c_float, C.c_void_p]),
    "w2s_stage_zscore": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]),
    "w2s_debug_timestamps": (C.c_int, [C.c_void_p, C.c_void_p]),
    "w2s_dropout": (C.c_int, [C.c_void_p] * 4 + [C.c_int64, C.c_float, C.c_uint64, C.c_uint32, C.c_void_p]),
    "w2s_attn_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_uint32, C.c_void_p]),
    "w2s_attn_bwd": (C.c_int, [C.c_void_p] * 8 + [C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_uint32, C.c_void_p]),
    "w2s_tokens_fwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                 C.c_int, C.c_int, C.c_void_p]),
    "w2s_tokens_bwd": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_int,
                                 C.c_int, C.c_float, C.c_void_p]),
    "w2s_rows_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "w2s_head_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "w2s_ce_fwd_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "w2s_head_bwd": (C.c_int, [C.c_void_p] * 6 + [C.c_longlong, C.c_int, C.c_float, C.c_void_p]),
    "w2s_sumsq": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "w2s_absmax": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "w2s_ig_path_inputs": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_void_p, C.c_void_p]),
    "w2s_ig_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                    C.c_int, C.c_void_p]),
    "w2s_adamw_step": (C.c_int, [C.c_void_p] * 4 + [C.c_longlong, C.c_void_p] + [C.c_float] * 7
                       + [C.c_longlong, C.c_void_p, C.c_float, C.c_void_p]),
    "w2s_gen_conv": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 11 + [C.c_void_p]),
    "w2s_gen_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "w2s_gen_norm_consts": (C.c_int, [C.c_void_p] * 7 + [C.c_int] * 5 + [C.c_float, C.c_void_p]),
    "w2s_gen_affine_act": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 5 + [C.c_void_p]),
    "w2s_gen_rownorm": (C.c_int, [C.c_void_p] * 4 + [C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_gen_attn": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 5 + [C.c_float, C.c_uint64, C.c_uint32, C.c_void_p]),
    "w2s_gen_conv_dgrad": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 10 + [C.c_void_p]),
    "w2s_gen_conv_wgrad": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 11 + [C.c_void_p]),
    "w2s_gen_affine_act_bwd": (C.c_int, [C.c_void_p] * 9 + [C.c_int] * 5 + [C.c_void_p]),
    "w2s_gen_norm_bwd": (C.c_int, [C.c_void_p] * 10 + [C.c_int] * 4 + [C.c_float, C.c_void_p]),
    "w2s_gen_rownorm_bwd": (C.c_int, [C.c_void_p] * 8 + [C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "w2s_gen_attn_bwd": (C.c_int, [C.c_void_p] * 8 + [C.c_int] * 5 + [C.c_float, C.c_uint64, C.c_uint32, C.c_void_p]),
    "w2s_gen_bn_eval_bwd": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_float, C.c_void_p]),
    "w2s_gen_bn_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "w2s_gen_bn_update_running": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int,
                                            C.c_void_p]),
    "w2s_gen_dropout": (C.c_int, [C.c_void_p] * 3 + [C.c_longlong, C.c_float, C.c_uint64, C.c_uint32, C.c_void_p]),
    "w2s_gen_seq_stream_step": (C.c_int, [C.POINTER(SeqStreamDesc), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                          C.c_void_p]),
    "w2s_launch_count": (C.c_longlong, []),
    "w2s_profile_enable": (C.c_int, [C.c_int]),
    "w2s_profile_count": (C.c_int, []),
    "w2s_profile_get": (C.c_int, [C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_double),
                                  C.POINTER(C.c_double)]),
}

_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load the shared library (building it first if needed).  Raises RuntimeError on any failure."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise RuntimeError(f"{LIB_PATH} is missing; run `python -c 'import __graft_entry__ as g; g.build()'`")
        build()
    try:
        lib = C.CDLL(str(LIB_PATH))
    except OSError as e:  # no silent fallback
        raise RuntimeError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.w2s_abi_version() != ABI_VERSION:
        raise RuntimeError(f"ABI mismatch: library {lib.w2s_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, exc=RuntimeError) -> None:
    if rc != 0:
        msg = load().w2s_last_error().decode()
        raise exc(msg)
