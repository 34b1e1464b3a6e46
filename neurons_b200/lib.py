"""ctypes binding of libneurons_mm.so (the C ABI declared in include/neurons_mm.h).

There is deliberately no fallback: if the shared object is missing, or a compute call is made without an
sm_100 GPU, this raises -- the product path never routes through PyTorch eager or the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get("NMM_LIB", "libneurons_mm.so"))     # NMM_LIB: development variants only

NMM_MAX_LAYERS = 4
NMM_MAX_ATTN = 4
NMM_MAX_FRAMES = 32
NMM_F32, NMM_BF16, NMM_F32X3, NMM_F32X6 = 0, 1, 2, 3
EPI_STORE, EPI_RESIDUAL, EPI_GEGLU, EPI_OUTPUT = 0, 1, 2, 3
STATUS_NAMES = {0: "NMM_OK", -1: "NMM_ERR_BAD_ARG", -2: "NMM_ERR_UNSUPPORTED", -3: "NMM_ERR_WORKSPACE",
                -4: "NMM_ERR_CUDA", -5: "NMM_ERR_DEVICE"}


class NmmError(RuntimeError):
    def __init__(self, status: int, text: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {text}")
        self.status = status


class Shape(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("channels", C.c_int32), ("frames", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
        ("heads", C.c_int32), ("layers", C.c_int32), ("attn_blocks", C.c_int32), ("pos_enc", C.c_int32),
        ("max_len", C.c_int32), ("dtype", C.c_int32), ("eps_gn", C.c_float), ("eps_ln", C.c_float), ("ln_fold", C.c_int32),
        ("x_stride_b", C.c_int64), ("x_stride_c", C.c_int64), ("x_stride_f", C.c_int64),
        ("y_stride_b", C.c_int64), ("y_stride_c", C.c_int64), ("y_stride_f", C.c_int64),
    ]


class AttnParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("norm_w", "norm_b", "to_q", "to_k", "to_v", "to_out_w", "to_out_b", "pe")]


class LayerParams(C.Structure):
    _fields_ = [("attn", AttnParams * NMM_MAX_ATTN)] + [
        (n, C.c_void_p) for n in ("ff_norm_w", "ff_norm_b", "ff_proj_w", "ff_proj_b", "ff_out_w", "ff_out_b")]


class Params(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("gn_w", C.c_void_p), ("gn_b", C.c_void_p), ("proj_in_w", C.c_void_p),
                ("proj_in_b", C.c_void_p), ("layer", LayerParams * NMM_MAX_LAYERS), ("proj_out_w", C.c_void_p),
                ("proj_out_b", C.c_void_p)]


class SpatialShape(C.Structure):
    _fields_ = [("base", Shape), ("ctx_len", C.c_int32), ("ctx_dim", C.c_int32)]


class SpatialLayerParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "norm1_w", "norm1_b", "attn1_q", "attn1_k", "attn1_v", "attn1_out_w", "attn1_out_b", "norm2_w", "norm2_b", "attn2_q", "attn2_k",
        "attn2_v", "attn2_out_w", "attn2_out_b", "norm3_w", "norm3_b", "ff_proj_w", "ff_proj_b", "ff_out_w", "ff_out_b")]


class SpatialParams(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("gn_w", C.c_void_p), ("gn_b", C.c_void_p), ("proj_in_w", C.c_void_p), ("proj_in_b", C.c_void_p),
                ("layer", SpatialLayerParams * NMM_MAX_LAYERS), ("proj_out_w", C.c_void_p), ("proj_out_b", C.c_void_p)]


class DecoderAttnParams(C.Structure):
    _fields_ = [("dtype", C.c_int32)] + [(n, C.c_void_p) for n in ("gn_w", "gn_b", "to_q_w", "to_q_b", "to_k_w", "to_k_b", "to_v_w", "to_v_b",
                                                                    "to_out_w", "to_out_b")]


class KernelProfile(C.Structure):
    _fields_ = [("name", C.c_char_p), ("launches", C.c_uint64), ("total_ms", C.c_double), ("flops", C.c_double),
                ("bytes", C.c_double)]


PROFILE_KERNELS = 12
ABI_VERSION = 3

# name -> (restype, argtypes); must list every NMM_API symbol of include/neurons_mm.h (tests/test_abi.py checks)
_SP = C.POINTER(Shape)
_SSP = C.POINTER(SpatialShape)
SIGNATURES = {
    "nmm_abi_version": (C.c_int, []),
    "nmm_last_error": (C.c_char_p, []),
    "nmm_device_check": (C.c_int, []),
    "nmm_launch_count": (C.c_uint64, []),
    "nmm_set_option": (C.c_int, [C.c_int32, C.c_int64]),
    "nmm_get_option": (C.c_int64, [C.c_int32]),
    "nmm_profile_begin": (C.c_int, []),
    "nmm_profile_end": (C.c_int, [C.POINTER(KernelProfile), C.c_int32]),
    "nmm_validate": (C.c_int, [_SP]),
    "nmm_packed_params_bytes": (C.c_int, [_SP, C.POINTER(C.c_size_t)]),
    "nmm_workspace_bytes": (C.c_int, [_SP, C.POINTER(C.c_size_t)]),
    "nmm_pack_params": (C.c_int, [_SP, C.POINTER(Params), C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_forward": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_forward_stats": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nmm_packed_header": (C.c_int, [_SP, C.c_void_p, C.c_size_t]),
    "nmm_forward_stage": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p, C.c_void_p]),
    "nmm_groupnorm_stats": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_groupnorm_tokens": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_groupnorm_linear": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_size_t, C.c_void_p]),
    "nmm_groupnorm_workspace_bytes": (C.c_int, [_SP, C.POINTER(C.c_size_t)]),
    "nmm_inflated_groupnorm": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_inflated_groupnorm_sums": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                              C.c_void_p]),
    "nmm_groupnorm_sums": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_cfg_ddim_step": (C.c_int, [C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_double, C.c_double, C.c_void_p]),
    "nmm_layernorm_pe": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nmm_temporal_attention": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nmm_qkv_attention": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nmm_linear": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_void_p, _SP, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nmm_spatial_packed_params_bytes": (C.c_int, [_SSP, C.POINTER(C.c_size_t)]),
    "nmm_spatial_workspace_bytes": (C.c_int, [_SSP, C.POINTER(C.c_size_t)]),
    "nmm_spatial_pack_params": (C.c_int, [_SSP, C.POINTER(SpatialParams), C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_spatial_forward": (C.c_int, [_SSP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_decoder_attn_packed_bytes": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "nmm_decoder_attn_workspace_bytes": (C.c_int, [_SP, C.POINTER(C.c_size_t)]),
    "nmm_decoder_attn_pack": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(DecoderAttnParams), C.c_float, C.c_float, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_decoder_temporal_attention": (C.c_int, [_SP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nmm_spatial_forward_stats": (C.c_int, [_SSP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                            C.c_void_p]),
    "nmm_spatial_attention": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                        C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load libneurons_mm.so (built in-tree by `python -m neurons_b200.build`).  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m neurons_b200.build` "
            "(there is no PyTorch/CPU fallback for the motion-module path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the ABI and this binding disagree
        fn.restype = res
        fn.argtypes = args
    if lib.nmm_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libneurons_mm.so ABI version {lib.nmm_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        raise NmmError(status, load().nmm_last_error().decode("utf-8", "replace"))


def profile_begin():
    check(load().nmm_profile_begin())


def profile_end():
    """-> {kernel name: dict(launches, total_ms, flops, bytes)} for the launches since profile_begin()."""
    arr = (KernelProfile * PROFILE_KERNELS)()
    check(load().nmm_profile_end(arr, PROFILE_KERNELS))
    return {k.name.decode(): dict(launches=int(k.launches), total_ms=float(k.total_ms), flops=float(k.flops), bytes=float(k.bytes))
            for k in arr}


# nmm_option (include/neurons_mm.h)
(OPT_FUSED_MODULE, OPT_GN_FUSE, OPT_ATTN_FUSE, OPT_WIDE_TILE, OPT_GEMM_CLUSTER, OPT_GEMM_BLOCK_N, OPT_CHUNK_TOKENS, OPT_ATTN_VARIANT, OPT_FUSED_Y_STATS,
 OPT_FUSED_CLUSTER, OPT_SPATIAL_ATTN) = range(11)


def set_option(option: int, value: int):
    check(load().nmm_set_option(option, value))


def get_option(option: int) -> int:
    return int(load().nmm_get_option(option))


class options:
    """Context manager: `with lib.options({lib.OPT_FUSED_MODULE: 0}): ...` -- set run-time options, restore them on exit."""

    def __init__(self, values: dict):
        self.values = dict(values)
        self.saved = {}

    def __enter__(self):
        for k, v in self.values.items():
            self.saved[k] = get_option(k)
            set_option(k, v)
        return self

    def __exit__(self, *exc):
        for k, v in self.saved.items():
            set_option(k, v)
        return False


def launch_count() -> int:
    return int(load().nmm_launch_count())
