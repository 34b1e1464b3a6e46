"""Host-side mirror of the reference's spatial transformer (SURVEY 8(f) N3), backed by libneurons_mm.so.

Reference interface mirrored:
    Transformer3DModel(num_attention_heads, attention_head_dim, in_channels, num_layers=1, ..., cross_attention_dim, ...,
                       unet_use_cross_frame_attention, unet_use_temporal_attention)
        .forward(hidden_states[b,c,f,h,w], encoder_hidden_states=None, timestep=None, return_dict=True)
                                                                    /root/reference/animatediff/models/attention.py:31-148
    BasicTransformerBlock                                           :151-300
called by the CrossAttn blocks right before the motion module (unet_blocks.py:273,409,509,752, `.sample`).

The mirror classes carry the SAME parameter names / shapes as the reference (`norm`, `proj_in` (1x1 Conv2d), `transformer_blocks.L.
{norm1, attn1.{to_q,to_k,to_v,to_out.0}, norm2, attn2.{...}, norm3, ff.net.0.proj, ff.net.2}`, `proj_out`), so SD-1.5 UNet checkpoints
load unchanged.  `patch_spatial(model)` rebinds `forward` on reference instances already inside a UNet3DConditionModel /
SparseControlNetModel.  As with the motion module the sub-modules are parameter containers: all arithmetic runs in the CUDA library and
there is no eager / CPU fallback.  Supported configuration = the one every NEURONS model uses (LayerNorm norms, plain self-attention
attn1, text cross-attention attn2, GEGLU, no attention bias, no mask); anything else raises.
"""
from __future__ import annotations

import ctypes as C
import sys
import types
from dataclasses import dataclass
from typing import Dict, Optional

import torch
from torch import nn

from . import lib as _lib
from . import ops
from .motion_module import FeedForward, _Engine


@dataclass(frozen=True)
class SpatialConfig:
    channels: int
    heads: int = 8
    layers: int = 1
    ctx_dim: int = 768
    # fp32 activations: True = every Linear on the tensor cores as 3 bf16 MMAs per product (NMM_F32X3; needs channels, ctx_dim % 64 == 0),
    # False (module flag `_nmm_fp32_fma` or env NMM_FP32_FMA=1) = the FMA-pipe GEMM (NMM_F32) and fp32 attention on the FMA pipe (no bf16
    # rounding anywhere; the tiled flash kernel at every UNet size, the one-warp-per-query checker kernel for small shapes).
    fp32_tc: bool = True


class Transformer3DModelOutput:
    """`.sample` holder (the reference's is a diffusers BaseOutput dataclass, attention.py:19-21)."""

    def __init__(self, sample: torch.Tensor):
        self.sample = sample


class CrossAttention(nn.Module):
    """Parameter container (diffusers CrossAttention: motion_module_new.py:119-176)."""

    def __init__(self, query_dim: int, cross_attention_dim: Optional[int] = None, heads: int = 8, dim_head: int = 64, bias: bool = False):
        super().__init__()
        if bias:
            raise NotImplementedError("neurons_b200: attention_bias=True is not used by any NEURONS config")
        inner = heads * dim_head
        kv_dim = cross_attention_dim if cross_attention_dim is not None else query_dim
        self.heads, self.scale = heads, dim_head ** -0.5
        self.sliceable_head_dim, self._slice_size = heads, None
        self.to_q = nn.Linear(query_dim, inner, bias=False)
        self.to_k = nn.Linear(kv_dim, inner, bias=False)
        self.to_v = nn.Linear(kv_dim, inner, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(inner, query_dim), nn.Dropout(0.0)])

    def set_attention_slice(self, slice_size):          # slicing trades memory for launches in the reference; scores are never materialised here
        if slice_size is not None and slice_size > self.sliceable_head_dim:
            raise ValueError(f"slice_size {slice_size} has to be smaller or equal to {self.sliceable_head_dim}.")
        self._slice_size = slice_size


class BasicTransformerBlock(nn.Module):
    def __init__(self, dim: int, num_attention_heads: int, attention_head_dim: int, cross_attention_dim: int):
        super().__init__()
        self.attn1 = CrossAttention(dim, None, num_attention_heads, attention_head_dim)
        self.norm1 = nn.LayerNorm(dim)
        self.attn2 = CrossAttention(dim, cross_attention_dim, num_attention_heads, attention_head_dim)
        self.norm2 = nn.LayerNorm(dim)
        self.ff = FeedForward(dim)
        self.norm3 = nn.LayerNorm(dim)


class Transformer3DModel(nn.Module):
    def __init__(self, num_attention_heads: int = 16, attention_head_dim: int = 88, in_channels: Optional[int] = None, num_layers: int = 1,
                 dropout: float = 0.0, norm_num_groups: int = 32, cross_attention_dim: Optional[int] = None, attention_bias: bool = False,
                 activation_fn: str = "geglu", num_embeds_ada_norm: Optional[int] = None, use_linear_projection: bool = False,
                 only_cross_attention: bool = False, upcast_attention: bool = False, unet_use_cross_frame_attention=None,
                 unet_use_temporal_attention=None):
        super().__init__()
        inner = num_attention_heads * attention_head_dim
        if (inner != in_channels or norm_num_groups != 32 or cross_attention_dim is None or attention_bias or activation_fn != "geglu"
                or num_embeds_ada_norm is not None or only_cross_attention or unet_use_cross_frame_attention or unet_use_temporal_attention
                or dropout != 0.0):
            raise NotImplementedError("neurons_b200: Transformer3DModel configuration not used by any NEURONS model")
        self.use_linear_projection = use_linear_projection
        self.num_attention_heads, self.attention_head_dim, self.in_channels = num_attention_heads, attention_head_dim, in_channels
        self.norm = nn.GroupNorm(num_groups=norm_num_groups, num_channels=in_channels, eps=1e-6, affine=True)
        self.proj_in = nn.Linear(in_channels, inner) if use_linear_projection else nn.Conv2d(in_channels, inner, kernel_size=1)
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(inner, num_attention_heads, attention_head_dim, cross_attention_dim) for _ in range(num_layers)])
        self.proj_out = nn.Linear(in_channels, inner) if use_linear_projection else nn.Conv2d(inner, in_channels, kernel_size=1)

    def forward(self, hidden_states, encoder_hidden_states=None, timestep=None, return_dict: bool = True):
        out = spatial_forward(self, hidden_states, encoder_hidden_states)
        return Transformer3DModelOutput(sample=out) if return_dict else (out,)


# ---- configuration / packing ---------------------------------------------------------------------------------------------------
def spatial_config_of(module: nn.Module) -> SpatialConfig:
    """Kernel configuration from a (reference or mirror) Transformer3DModel; raises on variants the library does not implement."""
    blocks = module.transformer_blocks
    b0 = blocks[0]
    channels = module.norm.num_channels
    for blk in blocks:
        if getattr(blk, "use_ada_layer_norm", False) or getattr(blk, "unet_use_cross_frame_attention", False) or \
                getattr(blk, "unet_use_temporal_attention", False) or getattr(blk, "only_cross_attention", False):
            raise NotImplementedError("neurons_b200: AdaLayerNorm / cross-frame / in-block temporal attention are not supported")
        if getattr(blk, "attn2", None) is None or getattr(blk, "norm2", None) is None:
            raise NotImplementedError("neurons_b200: a BasicTransformerBlock without text cross-attention is not supported")
        for attn in (blk.attn1, blk.attn2):
            if attn.to_q.bias is not None or getattr(attn, "group_norm", None) is not None or getattr(attn, "added_kv_proj_dim", None) is not None:
                raise NotImplementedError("neurons_b200: attention bias / group_norm / added_kv_proj_dim variants are not supported")
        if type(blk.ff.net[0]).__name__ != "GEGLU":
            raise NotImplementedError("neurons_b200: only the GEGLU feed-forward is supported")
    if module.norm.num_groups != 32 or b0.attn1.to_q.out_features != channels:
        raise NotImplementedError("neurons_b200: needs 32 GroupNorm groups and inner_dim == in_channels")
    heads = int(b0.attn1.heads)
    if channels // heads not in (40, 80, 160):
        raise NotImplementedError(f"neurons_b200: spatial attention head dim {channels // heads} (supported: 40, 80, 160)")
    return SpatialConfig(channels=channels, heads=heads, layers=len(blocks), ctx_dim=int(b0.attn2.to_k.in_features),
                         fp32_tc=not bool(module.__dict__.get("_nmm_fp32_fma", False)))


def _dtype_code(dt: torch.dtype, cfg: Optional["SpatialConfig"] = None) -> int:
    if dt == torch.float32:
        if cfg is not None and cfg.fp32_tc and cfg.channels % 64 == 0 and cfg.ctx_dim % 64 == 0 and ops._FP32_FMA_ENV in (None, "0"):
            return _lib.NMM_F32X3
        return _lib.NMM_F32
    if dt == torch.bfloat16:
        return _lib.NMM_BF16
    raise TypeError(f"neurons_mm supports float32 and bfloat16 activations, got {dt}")


def _shape(cfg: SpatialConfig, dtype: torch.dtype, B=1, F=1, H=1, W=1, ctx_len=1) -> _lib.SpatialShape:
    s = _lib.SpatialShape()
    b = s.base
    b.batch, b.channels, b.frames, b.height, b.width = B, cfg.channels, F, H, W
    b.heads, b.layers, b.attn_blocks, b.pos_enc, b.max_len = cfg.heads, cfg.layers, 1, 0, 0
    b.dtype, b.eps_gn, b.eps_ln, b.ln_fold = _dtype_code(dtype, cfg), ops.GN_EPS, ops.LN_EPS, 0
    s.ctx_len, s.ctx_dim = ctx_len, cfg.ctx_dim
    return s


def pack_spatial_params(cfg: SpatialConfig, tensors: Dict[str, torch.Tensor], compute_dtype: torch.dtype, device) -> torch.Tensor:
    """Pack a Transformer3DModel's parameters (state_dict keys, all on `device`, one dtype) into the library's layout."""
    lib = _lib.load()
    keep, src_dtype = [], None

    def ptr(key: str):
        nonlocal src_dtype
        t = tensors.get(key)
        if t is None:
            raise KeyError(f"neurons_mm.pack_spatial_params: missing parameter '{key}'")
        ops._require_cuda(t, key)
        t = t.detach()
        if not t.is_contiguous():
            t = t.contiguous()
        if src_dtype is None:
            src_dtype = t.dtype
        elif t.dtype != src_dtype:
            raise TypeError(f"neurons_mm.pack_spatial_params: mixed parameter dtypes ({src_dtype} vs {t.dtype} at '{key}')")
        keep.append(t)
        return t.data_ptr()

    p = _lib.SpatialParams()
    p.gn_w, p.gn_b = ptr("norm.weight"), ptr("norm.bias")
    p.proj_in_w, p.proj_in_b = ptr("proj_in.weight"), ptr("proj_in.bias")         # [C,C,1,1] conv weight == [C,C] row-major
    for l in range(cfg.layers):
        lp, b = p.layer[l], f"transformer_blocks.{l}."
        lp.norm1_w, lp.norm1_b = ptr(b + "norm1.weight"), ptr(b + "norm1.bias")
        lp.attn1_q, lp.attn1_k, lp.attn1_v = (ptr(b + f"attn1.to_{n}.weight") for n in "qkv")
        lp.attn1_out_w, lp.attn1_out_b = ptr(b + "attn1.to_out.0.weight"), ptr(b + "attn1.to_out.0.bias")
        lp.norm2_w, lp.norm2_b = ptr(b + "norm2.weight"), ptr(b + "norm2.bias")
        lp.attn2_q, lp.attn2_k, lp.attn2_v = (ptr(b + f"attn2.to_{n}.weight") for n in "qkv")
        lp.attn2_out_w, lp.attn2_out_b = ptr(b + "attn2.to_out.0.weight"), ptr(b + "attn2.to_out.0.bias")
        lp.norm3_w, lp.norm3_b = ptr(b + "norm3.weight"), ptr(b + "norm3.bias")
        lp.ff_proj_w, lp.ff_proj_b = ptr(b + "ff.net.0.proj.weight"), ptr(b + "ff.net.0.proj.bias")
        lp.ff_out_w, lp.ff_out_b = ptr(b + "ff.net.2.weight"), ptr(b + "ff.net.2.bias")
    p.proj_out_w, p.proj_out_b = ptr("proj_out.weight"), ptr("proj_out.bias")
    p.dtype = _dtype_code(src_dtype)
    s = _shape(cfg, compute_dtype)
    n = C.c_size_t()
    _lib.check(lib.nmm_spatial_packed_params_bytes(C.byref(s), C.byref(n)))
    packed = torch.empty(n.value, dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.nmm_spatial_pack_params(C.byref(s), C.byref(p), packed.data_ptr(), n.value, ops._stream_ptr(device)))
    del keep
    return packed


def spatial_forward_packed(x: torch.Tensor, encoder_hidden_states: torch.Tensor, packed: torch.Tensor, cfg: SpatialConfig,
                           shape_cache: Optional[dict] = None, y_sums: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y = Transformer3DModel(x, encoder_hidden_states).sample through nmm_spatial_forward: logical [B,C,F,H,W] over [B,F,C,H,W] storage
    (the strides attention.py:139's rearrange gives)."""
    ops._require_cuda(x, "hidden_states")
    ops._require_cuda(encoder_hidden_states, "encoder_hidden_states")
    x = ops._dense_hw(x)
    B, Cc, F, H, W = x.shape
    ehs = encoder_hidden_states
    if ehs.dim() != 3 or ehs.shape[0] != B or ehs.shape[2] != cfg.ctx_dim:
        raise ValueError(f"encoder_hidden_states must be [batch={B}, tokens, {cfg.ctx_dim}], got {tuple(ehs.shape)}")
    if ehs.dtype != x.dtype:
        raise TypeError(f"encoder_hidden_states dtype {ehs.dtype} != hidden_states dtype {x.dtype}")
    ehs = ehs.contiguous()
    out = torch.empty((B, F, Cc, H, W), dtype=x.dtype, device=x.device).permute(0, 2, 1, 3, 4)
    key = (x.shape, x.stride(), x.dtype, ehs.shape[1])
    hit = shape_cache.get(key) if shape_cache is not None else None
    lib = _lib.load()
    if hit is None:
        s = _shape(cfg, x.dtype, B, F, H, W, ehs.shape[1])
        b = s.base
        b.x_stride_b, b.x_stride_c, b.x_stride_f = x.stride(0), x.stride(1), x.stride(2)
        b.y_stride_b, b.y_stride_c, b.y_stride_f = out.stride(0), out.stride(1), out.stride(2)
        n = C.c_size_t()
        _lib.check(lib.nmm_spatial_workspace_bytes(C.byref(s), C.byref(n)))
        hit = (s, n.value)
        if shape_cache is not None:
            shape_cache[key] = hit
    s, ws_bytes = hit
    ws, ws_ptr = ops._aligned_ws(ws_bytes, x.device)
    with torch.cuda.device(x.device):
        if y_sums is not None:
            ops._check_sums(y_sums, x, "y_sums")
            _lib.check(lib.nmm_spatial_forward_stats(C.byref(s), x.data_ptr(), ehs.data_ptr(), out.data_ptr(), packed.data_ptr(), packed.numel(), ws_ptr,
                                                     ws_bytes, y_sums.data_ptr(), ops._stream_ptr(x.device)))
        else:
            _lib.check(lib.nmm_spatial_forward(C.byref(s), x.data_ptr(), ehs.data_ptr(), out.data_ptr(), packed.data_ptr(), packed.numel(), ws_ptr,
                                               ws_bytes, ops._stream_ptr(x.device)))
    return out


def spatial_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, kv_div: int = 1, x3: bool = False) -> torch.Tensor:
    """Per-stage entry (tests / micro-benchmarks): q [images, Lq, heads*dh], k / v [images / kv_div, Lkv, heads*dh] (last dim dense; row
    and image strides free) -> o [images, Lq, heads*dh].  nmm_spatial_attention.
    fp32 q, k, v (x3=False): fp32 throughout on the FMA pipe, the attention of the FMA mode -- the tiled flash kernel from 2^17 score elements
    (Lq * Lkv * images * heads) up, the checker kernel below; q, k, v need 16-byte alignment and strides in multiples of 4 for the tiled kernel.
    x3=True (fp32 q, k, v): the fp32-grade tensor-core kernel of the NMM_F32X3 mode -- q and k | v are converted to hi | lo planes here
    (like ops.linear(..., x3=True)); o is fp32."""
    for t, name in ((q, "q"), (k, "k"), (v, "v")):
        ops._require_cuda(t, name)
        if t.dim() != 3 or t.stride(2) != 1:
            raise ValueError(f"{name} must be [images, rows, channels] with dense channels")
    images, Lq, Cc = q.shape
    if k.shape != v.shape or k.stride() != v.stride() or k.shape[0] * kv_div != images or k.shape[2] != Cc:
        raise ValueError("k / v must share shape and strides, with images == kv images * kv_div")
    dt = _dtype_code(q.dtype)
    if x3:
        if q.dtype != torch.float32 or k.dtype != torch.float32 or v.dtype != torch.float32:
            raise TypeError("spatial_attention(x3=True) takes fp32 q, k, v")
        Lkv = k.shape[1]
        q = ops.split_planes(q.reshape(images * Lq, Cc)).view(images, Lq, 2 * Cc)                      # rows [hi q | lo q]
        kv = ops.split_planes(torch.cat([k, v], -1).reshape(-1, 2 * Cc)).view(-1, Lkv, 4 * Cc)        # rows [hi k | hi v | lo k | lo v]
        k, v, dt = kv[..., :Cc], kv[..., Cc:2 * Cc], _lib.NMM_F32X3
    o = torch.empty((images, Lq, Cc), dtype=torch.float32 if x3 else q.dtype, device=q.device)
    with torch.cuda.device(q.device):
        _lib.check(_lib.load().nmm_spatial_attention(dt, q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), q.stride(1), k.stride(1),
                                                     o.stride(1), q.stride(0), k.stride(0), o.stride(0), Lq, k.shape[1], heads, Cc // heads, images,
                                                     kv_div, ops._stream_ptr(q.device)))
    return o


# ---- engine + forward + patch ----------------------------------------------------------------------------------------------------
class _SpatialEngine(_Engine):
    def _tensors_of(self, module):
        return {k: v for k, v in module.named_parameters()}

    def _config_of(self, module):
        return spatial_config_of(module)

    def _pack(self, cfg, dev_tensors, x):
        return pack_spatial_params(cfg, dev_tensors, x.dtype, x.device)


def _engine_of(module: nn.Module) -> _SpatialEngine:
    eng = module.__dict__.get("_nmm_engine")
    if eng is None:
        eng = _SpatialEngine()
        module.__dict__["_nmm_engine"] = eng
    return eng


def spatial_forward(module: nn.Module, hidden_states: torch.Tensor, encoder_hidden_states: Optional[torch.Tensor]) -> torch.Tensor:
    """Transformer3DModel.forward on the B200 path (inference only)."""
    if hidden_states.dim() != 5:
        raise AssertionError(f"Expected hidden_states to have ndim=5, but got ndim={hidden_states.dim()}.")     # attention.py:97
    if encoder_hidden_states is None:
        raise ValueError("neurons_b200: Transformer3DModel needs encoder_hidden_states (the reference's `repeat` fails on None too, attention.py:100)")
    if not hidden_states.is_cuda:
        raise RuntimeError("neurons_b200: the spatial transformer runs on CUDA (sm_100) only; there is no CPU path")
    if torch.is_grad_enabled() and (hidden_states.requires_grad or any(p.requires_grad for p in module.parameters())):
        raise RuntimeError("neurons_b200: the spatial-transformer op is inference-only; call it under torch.no_grad()")
    eng = _engine_of(module)
    cfg, packed = eng.get(module, hidden_states)
    if not module.__dict__.get("_nmm_carry_stats", False):
        return spatial_forward_packed(hidden_states, encoder_hidden_states, packed, cfg, shape_cache=eng.shape_cache)
    # patch_spatial(model, carry_stats=True): proj_out's epilogue also emits the GroupNorm sums of the output; they ride on the tensor to
    # the motion module called next (patch(model, carry_stats=True)), which then skips its statistics pass (SURVEY 8(f) N1)
    from .motion_module import attach_sums
    B, _, F = hidden_states.shape[:3]
    y_sums = torch.empty((B * F * 32, 2), dtype=torch.float64, device=hidden_states.device)
    y = spatial_forward_packed(hidden_states, encoder_hidden_states, packed, cfg, shape_cache=eng.shape_cache, y_sums=y_sums)
    attach_sums(y, y_sums)
    return y


def _is_spatial_transformer(m: nn.Module) -> bool:
    return type(m).__name__ == "Transformer3DModel" and hasattr(m, "transformer_blocks") and hasattr(m, "proj_in")


def patch_spatial(model: nn.Module, carry_stats: bool = False) -> int:
    """Rebind `forward` on every Transformer3DModel inside `model` (reference instances included).  carry_stats=True: each call also emits
    the GroupNorm sums of its output for the motion module behind it (use with patch(model, carry_stats=True)).  Returns the number patched
    (16 in the SD-1.5 UNet3DConditionModel, 7 in SparseControlNetModel); unsupported configurations raise here."""
    n = 0
    for m in model.modules():
        if _is_spatial_transformer(m):
            spatial_config_of(m)
            m.__dict__["_nmm_carry_stats"] = bool(carry_stats)
            out_cls = getattr(sys.modules.get(type(m).__module__), "Transformer3DModelOutput", Transformer3DModelOutput)

            def _fwd(self, hidden_states, encoder_hidden_states=None, timestep=None, return_dict: bool = True, _out=out_cls):
                out = spatial_forward(self, hidden_states, encoder_hidden_states)
                return _out(sample=out) if return_dict else (out,)
            m.forward = types.MethodType(_fwd, m)
            n += 1
    return n
