"""ctypes binding of include/novic_b200.h (libnovic_b200.so, built in-tree by `make -C novic_b200/csrc`).

There is deliberately no fallback: if the shared library is missing, or no sm_100 device is present, the
decoder raises.  Nothing here imports the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

NOVIC_MAX_LAYERS = 16
NOVIC_MAX_BEAMS = 16

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libnovic_b200.so")
CSRC_DIR = os.path.join(_HERE, "csrc")


class NovicCfg(C.Structure):
    _fields_ = [
        ("embed_dim", C.c_int32), ("hidden_dim", C.c_int32), ("ffn_dim", C.c_int32), ("num_layers", C.c_int32),
        ("num_heads", C.c_int32), ("prefix_len", C.c_int32), ("vocab_size", C.c_int32), ("token_length", C.c_int32),
        ("strictly_causal", C.c_int32), ("num_end_loss", C.c_int32), ("ln_eps", C.c_float), ("label_smoothing", C.c_float),
    ]


_FP = C.c_void_p  # device pointers travel as integers


class NovicWeights(C.Structure):
    _fields_ = [
        ("embed_mlp", _FP), ("tok_embed", _FP), ("pos_embed", _FP), ("final_norm", _FP),
        ("in_proj", _FP * NOVIC_MAX_LAYERS), ("out_proj", _FP * NOVIC_MAX_LAYERS), ("linear1", _FP * NOVIC_MAX_LAYERS),
        ("linear2", _FP * NOVIC_MAX_LAYERS), ("norm1", _FP * NOVIC_MAX_LAYERS), ("norm2", _FP * NOVIC_MAX_LAYERS),
    ]


class NovicNoiseCfg(C.Structure):
    _fields_ = [
        ("scheme", C.c_int32), ("embed_dim", C.c_int32), ("vec_norm", C.c_float), ("angle_min", C.c_float),
        ("angle_max", C.c_float), ("angle_std", C.c_float), ("mix_ratio", C.c_float),
    ]


NOVIC_VIT_MAX_LAYERS = 48


class NovicVitCfg(C.Structure):
    _fields_ = [("image_size", C.c_int32), ("patch_size", C.c_int32), ("width", C.c_int32), ("layers", C.c_int32), ("heads", C.c_int32),
                ("mlp_dim", C.c_int32), ("out_dim", C.c_int32), ("ln_eps", C.c_float)]


class NovicVitWeights(C.Structure):
    _fields_ = [("conv1", _FP), ("class_embedding", _FP), ("positional_embedding", _FP), ("ln_pre_w", _FP), ("ln_pre_b", _FP),
                ("ln_post_w", _FP), ("ln_post_b", _FP), ("proj", _FP)] + [
        (name, _FP * NOVIC_VIT_MAX_LAYERS) for name in ("ln1_w", "ln1_b", "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "ln2_w", "ln2_b",
                                                        "fc_w", "fc_b", "cproj_w", "cproj_b")]


class NovicSiglipCfg(C.Structure):
    _fields_ = [("image_size", C.c_int32), ("patch_size", C.c_int32), ("width", C.c_int32), ("layers", C.c_int32), ("heads", C.c_int32),
                ("mlp_dim", C.c_int32), ("ln_eps", C.c_float)]


class NovicSiglipWeights(C.Structure):
    _fields_ = [(name, _FP) for name in ("patch_w", "patch_b", "pos_embed", "norm_w", "norm_b", "pool_latent", "pool_q_w", "pool_q_b",
                                         "pool_kv_w", "pool_kv_b", "pool_proj_w", "pool_proj_b", "pool_norm_w", "pool_norm_b",
                                         "pool_fc1_w", "pool_fc1_b", "pool_fc2_w", "pool_fc2_b")] + [
        (name, _FP * NOVIC_VIT_MAX_LAYERS) for name in ("norm1_w", "norm1_b", "qkv_w", "qkv_b", "proj_w", "proj_b", "norm2_w", "norm2_b",
                                                        "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class NovicAdamW(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("weight_decay", C.c_float),
                ("max_grad_norm", C.c_float), ("step", C.c_int64)]


class NovicGuide(C.Structure):
    _fields_ = [("child_off", _FP), ("child_tok", _FP), ("child_node", _FP), ("num_nodes", C.c_int32), ("num_edges", C.c_int32),
                ("renorm", C.c_int32), ("child_bias", _FP)]


# name -> (restype, argtypes); every symbol include/novic_b200.h declares
SIGNATURES = {
    "novic_last_error": (C.c_char_p, []),
    "novic_version": (C.c_int, []),
    "novic_create": (C.c_int, [C.POINTER(NovicCfg), C.POINTER(C.c_void_p)]),
    "novic_destroy": (C.c_int, [C.c_void_p]),
    "novic_weight_bytes": (C.c_size_t, [C.c_void_p]),
    "novic_set_weights": (C.c_int, [C.c_void_p, C.POINTER(NovicWeights), C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "novic_generate_greedy": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_float, C.c_float, _FP, _FP, _FP, _FP, _FP, _FP,
                                        C.POINTER(C.c_int32), C.POINTER(NovicGuide), C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_generate_greedy_async": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_float, C.c_float, _FP, _FP, _FP, _FP, _FP, _FP,
                                              C.POINTER(NovicGuide), C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_generate_beam": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_int32, C.c_float, C.c_float, _FP, _FP, _FP,
                                      C.POINTER(C.c_int32), C.POINTER(NovicGuide), C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_loss_totals": (C.c_int, [_FP, _FP, _FP, C.c_int64, _FP, _FP, C.c_void_p]),
    "novic_forward": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_int32, _FP, _FP, _FP, C.c_int32, C.c_int32, _FP, _FP, _FP,
                                _FP, C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_forward_guided": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_int32, _FP, _FP, _FP, C.c_int32, _FP, _FP, _FP, _FP,
                                       C.POINTER(NovicGuide), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_score_targets": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_int32, _FP, _FP, C.c_int32, C.c_float, C.POINTER(NovicGuide), _FP,
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_train_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "novic_train_fwd_bwd": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_int32, _FP, _FP, _FP, C.c_int32, _FP, _FP, _FP, C.POINTER(NovicWeights),
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_train_fwd_bwd_ex": (C.c_int, [C.c_void_p, _FP, C.c_int64, C.c_int32, _FP, _FP, _FP, C.c_int32, _FP, _FP, _FP, C.POINTER(NovicWeights),
                                         C.c_void_p, C.c_size_t, C.c_void_p, C.c_int32, C.c_void_p]),
    "novic_adamw_scratch_bytes": (C.c_size_t, []),
    "novic_adamw_step": (C.c_int, [C.POINTER(NovicAdamW), _FP, _FP, _FP, _FP, C.c_int64, _FP, _FP, C.c_void_p, C.c_size_t, _FP, C.c_void_p]),
    "novic_vit_create": (C.c_int, [C.POINTER(NovicVitCfg), C.POINTER(C.c_void_p)]),
    "novic_vit_destroy": (C.c_int, [C.c_void_p]),
    "novic_vit_weight_bytes": (C.c_size_t, [C.c_void_p]),
    "novic_vit_set_weights": (C.c_int, [C.c_void_p, C.POINTER(NovicVitWeights), C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_vit_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64]),
    "novic_vit_encode": (C.c_int, [C.c_void_p, _FP, C.c_int64, _FP, C.c_int32, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_siglip_create": (C.c_int, [C.POINTER(NovicSiglipCfg), C.POINTER(C.c_void_p)]),
    "novic_siglip_set_weights": (C.c_int, [C.c_void_p, C.POINTER(NovicSiglipWeights), C.c_void_p, C.c_size_t, C.c_void_p]),
    "novic_set_dropout": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_uint64]),
    "novic_noise_apply": (C.c_int, [C.POINTER(NovicNoiseCfg), _FP, C.c_int64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "novic_noise_apply_predrawn": (C.c_int, [C.POINTER(NovicNoiseCfg), _FP, C.c_int64, _FP, _FP, _FP, _FP, C.c_void_p]),
    "novic_debug_gemm": (C.c_int, [_FP, _FP, _FP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "novic_debug_trace": (C.c_int, [C.POINTER(C.c_int64), C.c_int32]),
    "novic_debug_ws_offset": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_char_p, C.POINTER(C.c_size_t)]),
    "novic_debug_keep_classes": (C.c_int, [C.c_void_p, C.c_uint32]),
    "novic_debug_redzone": (C.c_int, [C.c_size_t]),
    "novic_debug_zones": (C.c_int64, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_uint64), C.c_int64]),
    "novic_debug_transpose_bf16": (C.c_int, [_FP, C.c_int64, C.c_int32, C.c_int32, _FP, C.c_int32, C.c_void_p]),
    "novic_debug_wgrad": (C.c_int, [_FP, C.c_int32, _FP, C.c_int32, C.c_int64, C.c_int32, _FP, C.c_void_p]),
    "novic_debug_wgrad_mn": (C.c_int, [_FP, C.c_int32, C.c_int32, _FP, C.c_int32, C.c_int32, C.c_int64, _FP, C.c_void_p]),
    "novic_debug_wgrad_splits": (C.c_int32, [C.c_int64, C.c_int64, C.c_int32]),
    "novic_debug_vit_gemm": (C.c_int, [_FP, _FP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _FP, _FP, C.c_int32, _FP,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "novic_debug_vit_attention": (C.c_int, [_FP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _FP, C.c_void_p]),
    "novic_debug_siglip_map_attention": (C.c_int, [_FP, _FP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _FP, C.c_void_p]),
    "novic_debug_vit_layernorm": (C.c_int, [_FP, C.c_int64, _FP, _FP, _FP, _FP, C.c_int32, _FP, C.c_int32, C.c_int32, C.c_float, _FP, _FP, C.c_int32,
                                            C.c_void_p]),
    "novic_kernel_timing": (C.c_int, [C.c_int32]),
    "novic_kernel_times": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "novic_launch_count": (C.c_int64, []),
    "novic_watchdog": (C.c_int, [C.POINTER(C.c_uint32)]),
    "novic_set_use_graphs": (C.c_int, [C.c_void_p, C.c_int32]),
}

KERNEL_CLASSES = ("embed_prep", "prefix_gemm", "qkv_gemm", "attention", "outproj_gemm", "ffn1_gemm", "ffn2_gemm", "logits_gemm",
                  "select", "other")

_lib = None


def build(force: bool = False) -> str:
    """Compile libnovic_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    if force and os.path.exists(LIB_PATH):
        os.remove(LIB_PATH)
    subprocess.run(["make", "-C", CSRC_DIR], check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(f"build did not produce {LIB_PATH}")
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C {CSRC_DIR}` (or __graft_entry__.build()). "
                "novic_b200 has no CPU or PyTorch fallback path.")
        handle = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)  # raises AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


class NovicError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().novic_last_error()
        raise NovicError(msg.decode("utf-8", "replace") if msg else f"novic_b200 call failed with code {rc}")
