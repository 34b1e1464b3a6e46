"""Tensor-level wrappers over the C ABI: PyTorch supplies device memory and the stream, nothing else.

`torch.ops.neurons_mm.forward` is the drop-in custom op for VanillaTemporalModule.forward
(/root/reference/animatediff/models/motion_module.py:77-82); it is registered for the CUDA dispatch key only --
there is no CPU kernel and no autograd formula (the reference calls the module under torch.no_grad(),
animatediff/pipelines/pipeline_neuroclips.py:320).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import lib as _lib

GN_EPS = 1e-6   # motion_module.py:109
LN_EPS = 1e-5   # nn.LayerNorm default


@dataclass(frozen=True)
class ModuleConfig:
    """The hyper-parameters that reach the kernels (motion_module.py:49-60)."""
    channels: int
    heads: int = 8
    layers: int = 1
    attn_blocks: int = 2
    pos_enc: bool = True
    max_len: int = 24
    # bf16 mode: fold the LayerNorms into the QKV / GEGLU GEMMs (3 launches and one fp32 read of the residual fewer per call).
    # Measured on B200 it is slower (it moves work into the GEMM epilogue, which is the bottleneck: 8.5 vs 7.6 ms/step), so the
    # default keeps the separate, exactly-LayerNorm kernel; NMM_LN_FOLD=1 / ln_fold=True enables it (kept as a tested option).
    ln_fold: bool = False
    # fp32 activations: True = every Linear on the tensor cores as 3 bf16 MMAs per product (NMM_F32X3; needs channels % 64 == 0,
    # other widths use the FMA path); False (or env NMM_FP32_FMA=1) = the fp32 FMA-pipe GEMM (NMM_F32), kept as the checker.
    fp32_tc: bool = True
    # fp32 activations, exact: 6 bf16 MMAs per product over three-plane splits (NMM_F32X6; channels % 64 == 0), as accurate as the FMA
    # path; other widths use the FMA path, which is exact too.  Module flag `_nmm_fp32_exact` or env NMM_FP32_EXACT=1.
    fp32_exact: bool = False


_FP32_FMA_ENV = os.environ.get("NMM_FP32_FMA")     # read ONCE at import (pack and forward must agree on the mode)
_FP32_EXACT_ENV = os.environ.get("NMM_FP32_EXACT")


def fp32_exact_selected(module) -> bool:
    """Is the fp32-exact mode selected for this module (flag `_nmm_fp32_exact` or env NMM_FP32_EXACT=1)?  Raises when the FMA mode is
    selected for it too (flag `_nmm_fp32_fma` or env NMM_FP32_FMA=1): both are exact, and the choice between them is not made silently."""
    exact = bool(module.__dict__.get("_nmm_fp32_exact", False)) or _FP32_EXACT_ENV not in (None, "0")
    fma = bool(module.__dict__.get("_nmm_fp32_fma", False)) or _FP32_FMA_ENV not in (None, "0")
    if exact and fma:
        raise ValueError("neurons_b200: both the fp32-exact tensor-core mode (_nmm_fp32_exact / NMM_FP32_EXACT) and the FMA mode "
                         "(_nmm_fp32_fma / NMM_FP32_FMA) are selected for this module; select one")
    return exact


def _dtype_code(dt: torch.dtype, cfg: Optional["ModuleConfig"] = None) -> int:
    if dt == torch.float32:
        if cfg is not None and cfg.fp32_exact:
            return _lib.NMM_F32X6 if cfg.channels % 64 == 0 else _lib.NMM_F32
        if cfg is not None and cfg.fp32_tc and cfg.channels % 64 == 0 and _FP32_FMA_ENV in (None, "0"):
            return _lib.NMM_F32X3
        return _lib.NMM_F32
    if dt == torch.bfloat16:
        return _lib.NMM_BF16
    raise TypeError(f"neurons_mm supports float32 and bfloat16 activations, got {dt}")


_LN_FOLD_ENV = os.environ.get("NMM_LN_FOLD")       # read ONCE at import: the packed layout depends on it (pack and forward must agree)


def _ln_fold(cfg: "ModuleConfig") -> int:
    return int(bool(cfg.ln_fold) if _LN_FOLD_ENV is None else _LN_FOLD_ENV != "0")


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"neurons_mm: `{name}` must be a CUDA tensor (there is no CPU implementation of this path)")


def make_shape(cfg: ModuleConfig, x: torch.Tensor, y: Optional[torch.Tensor] = None, stage: bool = False) -> _lib.Shape:
    """nmm_shape of a module call.  stage=True (per-stage entry points): fp32 tensors are plain fp32 (NMM_F32), never the hi | lo
    plane format of the whole-module NMM_F32X3 mode."""
    if x.dim() != 5:
        # same invariant and message as the reference, motion_module.py:135
        raise AssertionError(f"Expected hidden_states to have ndim=5, but got ndim={x.dim()}.")
    B, Cc, F, H, W = x.shape
    s = _lib.Shape()
    s.batch, s.channels, s.frames, s.height, s.width = B, Cc, F, H, W
    s.heads, s.layers, s.attn_blocks = cfg.heads, cfg.layers, cfg.attn_blocks
    s.pos_enc, s.max_len = int(cfg.pos_enc), cfg.max_len
    s.dtype = _dtype_code(x.dtype, None if stage else cfg)
    s.eps_gn, s.eps_ln = GN_EPS, LN_EPS
    s.ln_fold = _ln_fold(cfg)
    s.x_stride_b, s.x_stride_c, s.x_stride_f = x.stride(0), x.stride(1), x.stride(2)
    if y is not None:
        s.y_stride_b, s.y_stride_c, s.y_stride_f = y.stride(0), y.stride(1), y.stride(2)
    else:   # [B,F,C,H,W] storage, like the reference's output (motion_module.py:153-156)
        s.y_stride_b, s.y_stride_c, s.y_stride_f = F * Cc * H * W, H * W, Cc * H * W
    return s


def _dense_hw(x: torch.Tensor) -> torch.Tensor:
    """The kernels take arbitrary (b, c, f) strides but need dense (h, w)."""
    W = x.shape[4]
    if (x.shape[4] == 1 or x.stride(4) == 1) and (x.shape[3] == 1 or x.stride(3) == W):
        return x
    return x.contiguous()


def packed_params_bytes(cfg: ModuleConfig, dtype: torch.dtype, frames: int = 1) -> int:
    s = _lib.Shape()
    s.batch = s.height = s.width = 1
    s.frames = frames
    s.channels, s.heads, s.layers, s.attn_blocks = cfg.channels, cfg.heads, cfg.layers, cfg.attn_blocks
    s.pos_enc, s.max_len, s.dtype = int(cfg.pos_enc), cfg.max_len, _dtype_code(dtype, cfg)
    s.eps_gn, s.eps_ln, s.ln_fold = GN_EPS, LN_EPS, _ln_fold(cfg)
    n = C.c_size_t()
    _lib.check(_lib.load().nmm_packed_params_bytes(C.byref(s), C.byref(n)))
    return n.value


def param_key(l: int, i: Optional[int], leaf: str) -> str:
    base = f"temporal_transformer.transformer_blocks.{l}."
    return base + (f"attention_blocks.{i}." if i is not None else "") + leaf


def pack_params(cfg: ModuleConfig, tensors: Dict[str, torch.Tensor], compute_dtype: torch.dtype, device) -> torch.Tensor:
    """Pack a module's parameters (state_dict-style keys, all on `device`, all fp32 or all bf16) into the
    library's layout.  `tensors` may also hold '...attention_blocks.I.pos_encoder.pe' buffers ([1,max_len,C])."""
    lib = _lib.load()
    src_dtype = None
    keep = []

    def ptr(key: str, required: bool = True):
        nonlocal src_dtype
        t = tensors.get(key)
        if t is None:
            if required:
                raise KeyError(f"neurons_mm.pack_params: missing parameter '{key}'")
            return None
        _require_cuda(t, key)
        t = t.detach()
        if not t.is_contiguous():
            t = t.contiguous()
        if src_dtype is None:
            src_dtype = t.dtype
        elif t.dtype != src_dtype:
            raise TypeError(f"neurons_mm.pack_params: mixed parameter dtypes ({src_dtype} vs {t.dtype} at '{key}')")
        keep.append(t)
        return t.data_ptr()

    p = _lib.Params()
    tt = "temporal_transformer."
    p.gn_w, p.gn_b = ptr(tt + "norm.weight"), ptr(tt + "norm.bias")
    p.proj_in_w, p.proj_in_b = ptr(tt + "proj_in.weight"), ptr(tt + "proj_in.bias")
    for l in range(cfg.layers):
        lp = p.layer[l]
        for i in range(cfg.attn_blocks):
            ap = lp.attn[i]
            ap.norm_w, ap.norm_b = ptr(param_key(l, None, f"norms.{i}.weight")), ptr(param_key(l, None, f"norms.{i}.bias"))
            ap.to_q, ap.to_k, ap.to_v = (ptr(param_key(l, i, f"to_{n}.weight")) for n in "qkv")
            ap.to_out_w, ap.to_out_b = ptr(param_key(l, i, "to_out.0.weight")), ptr(param_key(l, i, "to_out.0.bias"))
            ap.pe = ptr(param_key(l, i, "pos_encoder.pe"), required=False) if cfg.pos_enc else None
        lp.ff_norm_w, lp.ff_norm_b = ptr(param_key(l, None, "ff_norm.weight")), ptr(param_key(l, None, "ff_norm.bias"))
        lp.ff_proj_w, lp.ff_proj_b = ptr(param_key(l, None, "ff.net.0.proj.weight")), ptr(param_key(l, None, "ff.net.0.proj.bias"))
        lp.ff_out_w, lp.ff_out_b = ptr(param_key(l, None, "ff.net.2.weight")), ptr(param_key(l, None, "ff.net.2.bias"))
    p.proj_out_w, p.proj_out_b = ptr(tt + "proj_out.weight"), ptr(tt + "proj_out.bias")
    p.dtype = _dtype_code(src_dtype)

    nbytes = packed_params_bytes(cfg, compute_dtype)
    packed = torch.empty(nbytes, dtype=torch.uint8, device=device)
    s = _lib.Shape()
    s.batch = s.frames = s.height = s.width = 1
    s.channels, s.heads, s.layers, s.attn_blocks = cfg.channels, cfg.heads, cfg.layers, cfg.attn_blocks
    s.pos_enc, s.max_len, s.dtype = int(cfg.pos_enc), cfg.max_len, _dtype_code(compute_dtype, cfg)
    s.eps_gn, s.eps_ln, s.ln_fold = GN_EPS, LN_EPS, _ln_fold(cfg)
    with torch.cuda.device(device):
        _lib.check(lib.nmm_pack_params(C.byref(s), C.byref(p), packed.data_ptr(), nbytes, _stream_ptr(device)))
    del keep
    return packed


def _aligned_ws(nbytes: int, device):
    """Workspace buffer whose start is 1024-byte aligned (the caching allocator only guarantees 512)."""
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    ptr = (buf.data_ptr() + 1023) // 1024 * 1024
    return buf, ptr


def workspace_bytes(shape: _lib.Shape) -> int:
    n = C.c_size_t()
    _lib.check(_lib.load().nmm_workspace_bytes(C.byref(shape), C.byref(n)))
    return n.value


def _check_sums(t: torch.Tensor, x: torch.Tensor, name: str):
    B, _, F = x.shape[:3]
    if t.dtype != torch.float64 or t.shape != (B * F * 32, 2) or not t.is_contiguous() or t.device != x.device:
        raise ValueError(f"{name} must be a contiguous float64 [{B * F * 32}, 2] tensor on {x.device} (sum, sum of squares per (b, f, group))")


def forward_packed(x: torch.Tensor, packed: torch.Tensor, cfg: ModuleConfig, out: Optional[torch.Tensor] = None,
                   shape_cache: Optional[dict] = None, stage: Optional[int] = None, x_sums: Optional[torch.Tensor] = None,
                   y_sums: Optional[torch.Tensor] = None):
    """y = module(x) through nmm_forward.  Returns logical [B,C,F,H,W] over [B,F,C,H,W] storage.
    `shape_cache` (optional dict owned by the caller) memoises the validated nmm_shape + workspace size per input geometry.
    `stage` (tests): also return the fused kernel's fp32 [N, C] residual-stream snapshot after that stage (nmm_forward_stage).
    `x_sums` / `y_sums` (float64 [B*F*32, 2]): GroupNorm statistics handed in for x / written for y (nmm_forward_stats, SURVEY 8(f) N1)."""
    _require_cuda(x, "x")
    _require_cuda(packed, "packed")
    x = _dense_hw(x)
    B, Cc, F, H, W = x.shape
    if out is None:
        out = torch.empty((B, F, Cc, H, W), dtype=x.dtype, device=x.device).permute(0, 2, 1, 3, 4)
    key = (x.shape, x.stride(), out.stride(), x.dtype) if shape_cache is not None else None
    hit = shape_cache.get(key) if shape_cache is not None else None
    if hit is None:
        shape = make_shape(cfg, x, out)
        _lib.check(_lib.load().nmm_validate(C.byref(shape)))
        hit = (shape, workspace_bytes(shape))
        if shape_cache is not None:
            shape_cache[key] = hit
    shape, ws_bytes = hit
    ws, ws_ptr = _aligned_ws(ws_bytes, x.device)
    lib = _lib.load()
    if stage is not None:
        stage_out = torch.empty((B * F * H * W, Cc), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.nmm_forward_stage(C.byref(shape), x.data_ptr(), out.data_ptr(), packed.data_ptr(), packed.numel(), ws_ptr, ws_bytes,
                                             int(stage), stage_out.data_ptr(), _stream_ptr(x.device)))
        return out, stage_out
    if x_sums is not None or y_sums is not None:
        if x_sums is not None:
            _check_sums(x_sums, x, "x_sums")
        if y_sums is not None:
            _check_sums(y_sums, x, "y_sums")
        with torch.cuda.device(x.device):
            _lib.check(lib.nmm_forward_stats(C.byref(shape), x.data_ptr(), out.data_ptr(), packed.data_ptr(), packed.numel(), ws_ptr, ws_bytes,
                                             x_sums.data_ptr() if x_sums is not None else None,
                                             y_sums.data_ptr() if y_sums is not None else None, _stream_ptr(x.device)))
        return out
    if x.device.index != torch.cuda.current_device():
        with torch.cuda.device(x.device):
            _lib.check(lib.nmm_forward(C.byref(shape), x.data_ptr(), out.data_ptr(), packed.data_ptr(), packed.numel(), ws_ptr,
                                       ws_bytes, _stream_ptr(x.device)))
    else:
        _lib.check(lib.nmm_forward(C.byref(shape), x.data_ptr(), out.data_ptr(), packed.data_ptr(), packed.numel(), ws_ptr,
                                   ws_bytes, _stream_ptr(x.device)))
    return out


def packed_header(cfg: ModuleConfig, dtype: torch.dtype) -> bytes:
    """The 64-byte header nmm_pack_params writes for (cfg, dtype): compare with bytes(packed[:64].cpu())."""
    s = _lib.Shape()
    s.batch = s.frames = s.height = s.width = 1
    s.channels, s.heads, s.layers, s.attn_blocks = cfg.channels, cfg.heads, cfg.layers, cfg.attn_blocks
    s.pos_enc, s.max_len, s.dtype = int(cfg.pos_enc), cfg.max_len, _dtype_code(dtype, cfg)
    s.eps_gn, s.eps_ln, s.ln_fold = GN_EPS, LN_EPS, _ln_fold(cfg)
    buf = C.create_string_buffer(64)
    _lib.check(_lib.load().nmm_packed_header(C.byref(s), buf, 64))
    return buf.raw


# ---- torch.library registration: torch.ops.neurons_mm.forward ---------------------------------------------------
_LIBRARY = torch.library.Library("neurons_mm", "DEF")
_LIBRARY.define("forward(Tensor x, Tensor packed, int channels, int heads, int layers, int attn_blocks, bool pos_enc, int max_len) -> Tensor")


def _forward_cuda(x, packed, channels, heads, layers, attn_blocks, pos_enc, max_len):
    return forward_packed(x, packed, ModuleConfig(channels, heads, layers, attn_blocks, pos_enc, max_len))


def _forward_meta(x, packed, channels, heads, layers, attn_blocks, pos_enc, max_len):
    B, Cc, F, H, W = x.shape
    return x.new_empty((B, F, Cc, H, W)).permute(0, 2, 1, 3, 4)


_LIBRARY.impl("forward", _forward_cuda, "CUDA")
_LIBRARY.impl("forward", _forward_meta, "Meta")


# ---- per-stage wrappers (kernel-level parity tests, micro-benchmarks) --------------------------------------------
def _tokens(cfg: ModuleConfig, x: torch.Tensor):
    B, Cc, F, H, W = x.shape
    return B * F * H * W


def groupnorm_stats(cfg: ModuleConfig, x: torch.Tensor):
    x = _dense_hw(x)
    shape = make_shape(cfg, x, stage=True)
    B, F = x.shape[0], x.shape[2]
    mean = torch.empty(B * F * 32, dtype=torch.float32, device=x.device)
    rstd = torch.empty_like(mean)
    ws_bytes = workspace_bytes(shape)
    ws, ws_ptr = _aligned_ws(ws_bytes, x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().nmm_groupnorm_stats(C.byref(shape), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), ws_ptr,
                                                   ws_bytes, _stream_ptr(x.device)))
    return mean.view(B * F, 32), rstd.view(B * F, 32)


def groupnorm_tokens(cfg: ModuleConfig, x: torch.Tensor, gn_w: torch.Tensor, gn_b: torch.Tensor) -> torch.Tensor:
    x = _dense_hw(x)
    shape = make_shape(cfg, x, stage=True)
    tok = torch.empty((_tokens(cfg, x), cfg.channels), dtype=x.dtype, device=x.device)
    ws_bytes = workspace_bytes(shape)
    ws, ws_ptr = _aligned_ws(ws_bytes, x.device)
    gn_w, gn_b = gn_w.float().contiguous(), gn_b.float().contiguous()
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().nmm_groupnorm_tokens(C.byref(shape), x.data_ptr(), gn_w.data_ptr(), gn_b.data_ptr(), tok.data_ptr(),
                                                    ws_ptr, ws_bytes, _stream_ptr(x.device)))
    return tok


def groupnorm_linear(cfg: ModuleConfig, x: torch.Tensor, gn_w: torch.Tensor, gn_b: torch.Tensor, weight: torch.Tensor,
                     bias: Optional[torch.Tensor]) -> torch.Tensor:
    """GroupNorm + token re-layout + Linear in one tensor-core kernel (bf16): fp32 [N, C_out].  motion_module.py:142-145."""
    x = _dense_hw(x)
    shape = make_shape(cfg, x, stage=True)
    c_out = weight.shape[0]
    h = torch.empty((_tokens(cfg, x), c_out), dtype=torch.float32, device=x.device)
    ws_bytes = workspace_bytes(shape)
    ws, ws_ptr = _aligned_ws(ws_bytes, x.device)
    gn_w, gn_b = gn_w.float().contiguous(), gn_b.float().contiguous()
    weight = weight.to(x.dtype).contiguous()
    bias = bias.float().contiguous() if bias is not None else None
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().nmm_groupnorm_linear(C.byref(shape), x.data_ptr(), gn_w.data_ptr(), gn_b.data_ptr(), weight.data_ptr(), c_out,
                                                    bias.data_ptr() if bias is not None else None, h.data_ptr(), ws_ptr, ws_bytes,
                                                    _stream_ptr(x.device)))
    return h


def groupnorm_sums(x: torch.Tensor) -> torch.Tensor:
    """(sum, sum of squares) of x [b, c, f, h, w] per (b, f, GroupNorm group): float64 [B*F*32, 2] (nmm_groupnorm_sums)."""
    _require_cuda(x, "x")
    x = _dense_hw(x)
    shape = make_shape(ModuleConfig(x.shape[1], heads=1, pos_enc=False), x, stage=True)
    n = C.c_size_t()
    lib = _lib.load()
    _lib.check(lib.nmm_groupnorm_workspace_bytes(C.byref(shape), C.byref(n)))
    ws, ws_ptr = _aligned_ws(n.value, x.device)
    sums = torch.empty((x.shape[0] * x.shape[2] * 32, 2), dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.nmm_groupnorm_sums(C.byref(shape), x.data_ptr(), sums.data_ptr(), ws_ptr, n.value, _stream_ptr(x.device)))
    return sums


def inflated_groupnorm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-5, silu: bool = False,
                       out: Optional[torch.Tensor] = None, sums: Optional[torch.Tensor] = None) -> torch.Tensor:
    """InflatedGroupNorm(32, C, eps) of x [b, c, f, h, w] (+ SiLU): animatediff/models/resnet.py:21-29 (+ :185-186 / :198).
    Returns a contiguous [b, c, f, h, w] tensor (what the reference's rearrange-back produces) unless `out` is given.
    `sums`: the statistics of x from its producer (forward_packed(..., y_sums=...)): the statistics pass over x is skipped."""
    if not x.is_cuda:
        raise RuntimeError("neurons_b200.ops.inflated_groupnorm: CUDA tensors only (there is no CPU path)")
    x = _dense_hw(x)
    y = out if out is not None else torch.empty(x.shape, dtype=x.dtype, device=x.device)
    if y.shape != x.shape or y.dtype != x.dtype or _dense_hw(y) is not y:
        raise ValueError("out must have the shape / dtype of x and dense (h, w)")
    shape = make_shape(ModuleConfig(x.shape[1], heads=1, pos_enc=False), x, y, stage=True)
    shape.eps_gn = eps
    n = C.c_size_t()
    lib = _lib.load()
    _lib.check(lib.nmm_groupnorm_workspace_bytes(C.byref(shape), C.byref(n)))
    ws, ws_ptr = _aligned_ws(n.value, x.device)
    w, b = weight.float().contiguous(), bias.float().contiguous()
    with torch.cuda.device(x.device):
        if sums is not None:
            _check_sums(sums, x, "sums")
            _lib.check(lib.nmm_inflated_groupnorm_sums(C.byref(shape), x.data_ptr(), y.data_ptr(), w.data_ptr(), b.data_ptr(), int(silu),
                                                       sums.data_ptr(), ws_ptr, n.value, _stream_ptr(x.device)))
        else:
            _lib.check(lib.nmm_inflated_groupnorm(C.byref(shape), x.data_ptr(), y.data_ptr(), w.data_ptr(), b.data_ptr(), int(silu), ws_ptr, n.value,
                                                  _stream_ptr(x.device)))
    return y


def qkv_attention(cfg: ModuleConfig, bfhw, tokens: torch.Tensor, wqkv: torch.Tensor) -> torch.Tensor:
    """QKV projection + temporal attention in one tensor-core kernel (bf16): ctx [N, C].  wqkv: [3C, C] = cat(to_q, to_k, to_v)."""
    B, F, H, W = bfhw
    shape = _shape_for_tokens(cfg, B, F, H, W, tokens.dtype)
    tokens = tokens.contiguous()
    wqkv = wqkv.to(tokens.dtype).contiguous()
    scratch = torch.empty_like(wqkv)
    ctx = torch.empty_like(tokens)
    with torch.cuda.device(tokens.device):
        _lib.check(_lib.load().nmm_qkv_attention(C.byref(shape), tokens.data_ptr(), wqkv.data_ptr(), scratch.data_ptr(), ctx.data_ptr(),
                                                 _stream_ptr(tokens.device)))
    return ctx


def cfg_ddim_step(latents: torch.Tensor, eps_uncond: torch.Tensor, eps_cond: Optional[torch.Tensor], guidance: float, alpha_t: float,
                  alpha_prev: float) -> torch.Tensor:
    """In-place fused classifier-free guidance + DDIM update on CUDA tensors (pipeline_neuroclips.py:478-483); returns `latents`."""
    if not latents.is_cuda:
        raise RuntimeError("neurons_b200.ops.cfg_ddim_step: CUDA tensors only (there is no CPU path)")
    if not latents.is_contiguous():
        raise ValueError("latents must be contiguous (updated in place)")
    eu = eps_uncond.to(latents.dtype).contiguous()
    ec = eps_cond.to(latents.dtype).contiguous() if eps_cond is not None else None
    if eu.shape != latents.shape or (ec is not None and ec.shape != latents.shape):
        raise ValueError("eps tensors must have the shape of latents")
    with torch.cuda.device(latents.device):
        _lib.check(_lib.load().nmm_cfg_ddim_step(_dtype_code(latents.dtype), latents.numel(), latents.data_ptr(), eu.data_ptr(),
                                                 ec.data_ptr() if ec is not None else None, float(guidance), float(alpha_t), float(alpha_prev),
                                                 _stream_ptr(latents.device)))
    return latents


def _shape_for_tokens(cfg: ModuleConfig, B: int, F: int, H: int, W: int, dtype: torch.dtype) -> _lib.Shape:
    s = _lib.Shape()
    s.batch, s.channels, s.frames, s.height, s.width = B, cfg.channels, F, H, W
    s.heads, s.layers, s.attn_blocks = cfg.heads, cfg.layers, cfg.attn_blocks
    s.pos_enc, s.max_len, s.dtype = int(cfg.pos_enc), cfg.max_len, _dtype_code(dtype)
    s.eps_gn, s.eps_ln, s.ln_fold = GN_EPS, LN_EPS, 0
    P = H * W
    s.x_stride_b, s.x_stride_c, s.x_stride_f = cfg.channels * F * P, F * P, P
    s.y_stride_b, s.y_stride_c, s.y_stride_f = F * cfg.channels * P, P, cfg.channels * P
    return s


def layernorm_pe(cfg: ModuleConfig, dims, h: torch.Tensor, w: torch.Tensor, b: torch.Tensor, pe: Optional[torch.Tensor],
                 out_dtype: torch.dtype) -> torch.Tensor:
    B, F, H, W = dims
    shape = _shape_for_tokens(cfg, B, F, H, W, out_dtype)
    h = h.float().contiguous()
    out = torch.empty(h.shape, dtype=out_dtype, device=h.device)
    w, b = w.float().contiguous(), b.float().contiguous()
    pe_ptr = None
    if pe is not None:
        pe = pe.float().contiguous()
        pe_ptr = pe.data_ptr()
    with torch.cuda.device(h.device):
        _lib.check(_lib.load().nmm_layernorm_pe(C.byref(shape), h.data_ptr(), w.data_ptr(), b.data_ptr(), pe_ptr, out.data_ptr(),
                                                _stream_ptr(h.device)))
    return out


def temporal_attention(cfg: ModuleConfig, dims, qkv: torch.Tensor) -> torch.Tensor:
    B, F, H, W = dims
    shape = _shape_for_tokens(cfg, B, F, H, W, qkv.dtype)
    qkv = qkv.contiguous()
    ctx = torch.empty((qkv.shape[0], cfg.channels), dtype=qkv.dtype, device=qkv.device)
    with torch.cuda.device(qkv.device):
        _lib.check(_lib.load().nmm_temporal_attention(C.byref(shape), qkv.data_ptr(), ctx.data_ptr(), _stream_ptr(qkv.device)))
    return ctx


def split_planes(t: torch.Tensor, planes: int = 2) -> torch.Tensor:
    """fp32 [rows, K] -> the NMM_F32X3 operand format (planes=2): bf16 [rows, 2K], row = hi plane | lo plane (t = hi + lo + O(2^-17 t)),
    or the NMM_F32X6 format (planes=3): bf16 [rows, 3K], row = hi | mid | lo, hi = bf16(t), mid = bf16(t - hi), lo = bf16(t - hi - mid)
    (each difference in fp32, where it is exact; t = hi + mid + lo + O(2^-24 t))."""
    if planes not in (2, 3):
        raise ValueError(f"split_planes: planes must be 2 or 3, got {planes}")
    r = t.float()
    out = []
    for _ in range(planes):
        p = r.to(torch.bfloat16)
        out.append(p)
        r = r - p.float()
    return torch.cat(out, dim=1).contiguous()


def merge_planes(t: torch.Tensor, planes: int = 2) -> torch.Tensor:
    k = t.shape[1] // planes
    out = t[:, :k].float()
    for i in range(1, planes):
        out = out + t[:, i * k:(i + 1) * k].float()
    return out


def linear(A: torch.Tensor, Wt: torch.Tensor, bias: Optional[torch.Tensor] = None, epilogue: int = _lib.EPI_STORE,
           h: Optional[torch.Tensor] = None, want_out: bool = True, cfg: Optional[ModuleConfig] = None,
           x: Optional[torch.Tensor] = None, x3: bool = False, x6: bool = False) -> Optional[torch.Tensor]:
    """D = A . Wt^T with a fused epilogue (see include/neurons_mm.h nmm_epilogue).  A: [M,K], Wt: [N,K].
    x3=True (fp32 A / Wt): the 3 x bf16 tensor-core mode -- operands are converted to hi | lo planes here, `out` is merged back to fp32.
    x6=True (fp32 A / Wt): the 6 x bf16 (fp32-exact) tensor-core mode, the same with hi | mid | lo planes."""
    _require_cuda(A, "A")
    A, Wt = A.contiguous(), Wt.contiguous()
    M, K = A.shape
    N = Wt.shape[0]
    dt = _dtype_code(A.dtype)
    if x3 and x6:
        raise ValueError("linear: x3 and x6 are exclusive")
    planes = 3 if x6 else 2 if x3 else 1
    if planes > 1:
        assert A.dtype == torch.float32 and Wt.dtype == torch.float32
        A, Wt, dt = split_planes(A, planes), split_planes(Wt, planes), (_lib.NMM_F32X6 if x6 else _lib.NMM_F32X3)
    bias_ptr = None
    if bias is not None:
        bias = bias.float().contiguous()
        bias_ptr = bias.data_ptr()
    out = None
    shape_ref = None
    x_ptr = y_ptr = None
    if epilogue == _lib.EPI_OUTPUT:
        x = _dense_hw(x)
        B, Cc, F, H, W = x.shape
        out = torch.empty((B, F, Cc, H, W), dtype=x.dtype, device=x.device).permute(0, 2, 1, 3, 4)
        shape = make_shape(cfg, x, out)
        shape.dtype = dt
        shape_ref = C.byref(shape)
        x_ptr, y_ptr = x.data_ptr(), out.data_ptr()
        out_ptr = None
    else:
        if want_out:
            out = torch.empty((M, (N // 2 if epilogue == _lib.EPI_GEGLU else N) * planes), dtype=A.dtype, device=A.device)
        out_ptr = out.data_ptr() if out is not None else None
    h_ptr = h.data_ptr() if h is not None else None
    with torch.cuda.device(A.device):
        _lib.check(_lib.load().nmm_linear(dt, epilogue, M, N, K, A.data_ptr(), Wt.data_ptr(), bias_ptr, h_ptr, out_ptr, shape_ref,
                                          x_ptr, y_ptr, _stream_ptr(A.device)))
    if planes > 1 and out is not None and epilogue != _lib.EPI_OUTPUT:
        out = merge_planes(out, planes)
    return out
