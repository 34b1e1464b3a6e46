"""Host-side mirror of the reference's motion-module interface, backed by libneurons_mm.so.

Reference interface mirrored (same names, arguments and error behaviour):
    get_motion_module(in_channels, motion_module_type, motion_module_kwargs)      animatediff/models/motion_module.py:37-45
    VanillaTemporalModule(in_channels, num_attention_heads=8, ...).forward(input_tensor, temb, encoder_hidden_states,
        attention_mask=None, anchor_frame_idx=None)                               :48-82
The module tree carries the SAME parameter names and shapes as the reference
(`temporal_transformer.{norm,proj_in,transformer_blocks.L.{attention_blocks.I.{to_q,to_k,to_v,to_out.0},norms.I,
ff.net.0.proj,ff.net.2,ff_norm},proj_out}`), so `motion_modules.*` checkpoints (animatediff/utils/util.py:107-121)
load with load_state_dict unchanged; `pos_encoder.pe` is a non-persistent buffer as in :239.

Two ways in:
  * build a UNet with these classes (get_motion_module is signature-compatible), or
  * `patch(model)`: rebind `forward` on every *reference* VanillaTemporalModule already inside a UNet3DConditionModel /
    SparseControlNetModel.  Parameters stay where they are, so load_weights, LoRA merging (which mutates
    `.weight.data` in place) and state_dict() keep working; call `invalidate(model)` after mutating weights post-first-call.

The sub-modules below are parameter containers: the arithmetic of the whole path runs in the CUDA library,
there is no eager PyTorch implementation here and none is ever dispatched to.
"""
from __future__ import annotations

import math
import types
from typing import Dict, Optional

import torch
from torch import nn

import os

from . import ops
from .ops import ModuleConfig

_WEIGHT_CHECK = os.environ.get("NMM_WEIGHT_CHECK", "0") not in ("", "0")      # debug: checksum the live parameters on every call


def zero_module(module: nn.Module) -> nn.Module:
    """Zero every parameter (reference: motion_module.py:18-22)."""
    with torch.no_grad():
        for p in module.parameters():
            p.zero_()
    return module


def get_motion_module(in_channels, motion_module_type: str, motion_module_kwargs: dict):
    if motion_module_type == "Vanilla":
        return VanillaTemporalModule(in_channels=in_channels, **motion_module_kwargs)
    raise ValueError          # same as the reference (:45)


def sinusoidal_table(d_model: int, max_len: int) -> torch.Tensor:
    """[1, max_len, d_model] fp32 table; formula of PositionalEncoding.__init__ (:234-238)."""
    pos = torch.arange(max_len, dtype=torch.float32).unsqueeze(1)
    freq = torch.exp(torch.arange(0, d_model, 2, dtype=torch.float32) * (-math.log(10000.0) / d_model))
    table = torch.zeros(1, max_len, d_model)
    table[0, :, 0::2] = torch.sin(pos * freq)
    table[0, :, 1::2] = torch.cos(pos * freq)
    return table


class PositionalEncoding(nn.Module):
    def __init__(self, d_model: int, dropout: float = 0.0, max_len: int = 24):
        super().__init__()
        self.register_buffer("pe", sinusoidal_table(d_model, max_len), persistent=False)


class VersatileAttention(nn.Module):
    """Parameter container for one temporal self-attention block (reference :246-329 + diffusers CrossAttention)."""

    def __init__(self, query_dim: int, heads: int, dim_head: int, attention_mode: str = "Temporal",
                 cross_attention_dim: Optional[int] = None, temporal_position_encoding: bool = False,
                 temporal_position_encoding_max_len: int = 24):
        super().__init__()
        assert attention_mode == "Temporal"                      # :256
        if cross_attention_dim is not None:
            raise NotImplementedError("neurons_b200: '*_Cross' temporal attention blocks are not used by any NEURONS config")
        inner = heads * dim_head
        self.attention_mode = attention_mode
        self.is_cross_attention = False
        self.heads = heads
        self.scale = dim_head ** -0.5
        self.sliceable_head_dim = heads      # unet.set_attention_slice walks modules exposing these (unet.py:265-314)
        self._slice_size = None
        self.to_q = nn.Linear(query_dim, inner, bias=False)
        self.to_k = nn.Linear(query_dim, inner, bias=False)
        self.to_v = nn.Linear(query_dim, inner, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(inner, query_dim), nn.Dropout(0.0)])
        self.pos_encoder = (PositionalEncoding(query_dim, 0.0, temporal_position_encoding_max_len)
                            if temporal_position_encoding else None)

    def set_attention_slice(self, slice_size):
        # slicing only trades memory for launches in the reference; the fused kernel never materialises the scores
        if slice_size is not None and slice_size > self.sliceable_head_dim:
            raise ValueError(f"slice_size {slice_size} has to be smaller or equal to {self.sliceable_head_dim}.")
        self._slice_size = slice_size


class GEGLU(nn.Module):
    def __init__(self, dim_in: int, dim_out: int):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)


class FeedForward(nn.Module):
    """Parameter container: net.0 = GEGLU(dim -> 4*dim), net.1 = Dropout(0), net.2 = Linear(4*dim -> dim)."""

    def __init__(self, dim: int, mult: int = 4):
        super().__init__()
        self.net = nn.ModuleList([GEGLU(dim, dim * mult), nn.Dropout(0.0), nn.Linear(dim * mult, dim)])


class TemporalTransformerBlock(nn.Module):
    def __init__(self, dim: int, num_attention_heads: int, attention_head_dim: int, attention_block_types,
                 temporal_position_encoding: bool, temporal_position_encoding_max_len: int):
        super().__init__()
        blocks, norms = [], []
        for name in attention_block_types:
            blocks.append(VersatileAttention(
                query_dim=dim, heads=num_attention_heads, dim_head=attention_head_dim,
                attention_mode=name.split("_")[0],
                cross_attention_dim=768 if name.endswith("_Cross") else None,
                temporal_position_encoding=temporal_position_encoding,
                temporal_position_encoding_max_len=temporal_position_encoding_max_len))
            norms.append(nn.LayerNorm(dim))
        self.attention_blocks = nn.ModuleList(blocks)
        self.norms = nn.ModuleList(norms)
        self.ff = FeedForward(dim)
        self.ff_norm = nn.LayerNorm(dim)


class TemporalTransformer3DModel(nn.Module):
    def __init__(self, in_channels: int, num_attention_heads: int, attention_head_dim: int, num_layers: int,
                 attention_block_types=("Temporal_Self", "Temporal_Self"), norm_num_groups: int = 32,
                 temporal_position_encoding: bool = False, temporal_position_encoding_max_len: int = 24):
        super().__init__()
        inner = num_attention_heads * attention_head_dim
        if inner != in_channels:
            raise NotImplementedError("neurons_b200: temporal_attention_dim_div != 1 (inner_dim != in_channels) is not supported")
        self.norm = nn.GroupNorm(num_groups=norm_num_groups, num_channels=in_channels, eps=1e-6, affine=True)
        self.proj_in = nn.Linear(in_channels, inner)
        self.transformer_blocks = nn.ModuleList([
            TemporalTransformerBlock(inner, num_attention_heads, attention_head_dim, attention_block_types,
                                     temporal_position_encoding, temporal_position_encoding_max_len)
            for _ in range(num_layers)])
        self.proj_out = nn.Linear(inner, in_channels)


class VanillaTemporalModule(nn.Module):
    def __init__(self, in_channels, num_attention_heads=8, num_transformer_block=2,
                 attention_block_types=("Temporal_Self", "Temporal_Self"), cross_frame_attention_mode=None,
                 temporal_position_encoding=False, temporal_position_encoding_max_len=24,
                 temporal_attention_dim_div=1, zero_initialize=True):
        super().__init__()
        self.temporal_transformer = TemporalTransformer3DModel(
            in_channels=in_channels,
            num_attention_heads=num_attention_heads,
            attention_head_dim=in_channels // num_attention_heads // temporal_attention_dim_div,
            num_layers=num_transformer_block,
            attention_block_types=attention_block_types,
            temporal_position_encoding=temporal_position_encoding,
            temporal_position_encoding_max_len=temporal_position_encoding_max_len,
        )
        if zero_initialize:
            zero_module(self.temporal_transformer.proj_out)

    def forward(self, input_tensor, temb=None, encoder_hidden_states=None, attention_mask=None, anchor_frame_idx=None):
        # temb, encoder_hidden_states (Temporal_Self blocks), attention_mask and anchor_frame_idx are ignored by the
        # reference too (:77-82, :210-217)
        return motion_forward(self, input_tensor)


# ---- engine: per-module packed-parameter cache + the call into the CUDA library ----------------------------------
def config_of(module: nn.Module) -> ModuleConfig:
    """Derive the kernel configuration from a (reference or mirror) VanillaTemporalModule's tree."""
    tt = module.temporal_transformer
    blocks = tt.transformer_blocks
    b0 = blocks[0]
    for blk in blocks:
        for attn in blk.attention_blocks:
            if getattr(attn, "is_cross_attention", False) or getattr(attn, "attention_mode", "Temporal") != "Temporal":
                raise NotImplementedError("neurons_b200: only 'Temporal_Self' attention blocks are supported")
            if getattr(attn, "group_norm", None) is not None or getattr(attn, "added_kv_proj_dim", None) is not None:
                raise NotImplementedError("neurons_b200: group_norm / added_kv_proj_dim attention variants are not supported")
            if getattr(attn, "upcast_attention", False) or getattr(attn, "upcast_softmax", False):
                pass      # softmax already runs in fp32 here
    a0 = b0.attention_blocks[0]
    channels = tt.norm.num_channels
    if tt.proj_in.out_features != channels:
        raise NotImplementedError("neurons_b200: inner_dim != in_channels is not supported")
    pos = getattr(a0, "pos_encoder", None)
    return ModuleConfig(channels=channels, heads=int(a0.heads), layers=len(blocks), attn_blocks=len(b0.attention_blocks),
                        pos_enc=pos is not None, max_len=int(pos.pe.shape[1]) if pos is not None else 0,
                        ln_fold=bool(module.__dict__.get("_nmm_ln_fold", False)),      # set by tests / experiments before the first call
                        fp32_tc=not bool(module.__dict__.get("_nmm_fp32_fma", False)),  # fp32 activations: tensor cores (3 x bf16) unless set
                        fp32_exact=ops.fp32_exact_selected(module))                       # fp32 activations: 6 x bf16 (exact), raises with the FMA flag


def _param_tensors(module: nn.Module) -> Dict[str, torch.Tensor]:
    out = {k: v for k, v in module.named_parameters()}
    out.update({k: v for k, v in module.named_buffers() if k.endswith("pos_encoder.pe")})
    return out


class _Engine:
    """Packed copy of one module's parameters.

    Cache key: (dtype, device) of the call + (data_ptr, _version) of every source tensor.  `_version` catches every in-place update
    made through the tensor itself (load_state_dict / copy_, optimizer steps, `p += d`); `data_ptr` catches replaced parameters
    (.to(), .half()).  What neither sees is a write through `.data` (`p.data += d`: the reference's LoRA merge,
    convert_lora_safetensor_to_diffusers.py:27-47, detaches the version counter): call `neurons_b200.invalidate(model)` after such
    a merge, or run with NMM_WEIGHT_CHECK=1 (debug: a device-side checksum of all parameters is compared on every call, at the cost
    of one reduction + host sync per call) to be told when it happened."""

    def __init__(self):
        self.key = None
        self.packed = None
        self.cfg = None
        self.tensors = None      # name -> tensor, collected once (module.to() / .data updates keep the same objects)
        self.shape_cache = {}    # (shape, strides, dtype) -> (nmm_shape struct, workspace bytes)
        self.checksum = None

    @staticmethod
    def _key(x, tensors):
        return (x.dtype, x.device) + tuple((t.data_ptr(), t._version) for t in tensors.values())

    @staticmethod
    def _flags(module):
        # per-module mode switches that change the packed layout: part of the key, so flipping one re-packs instead of being ignored
        return (bool(module.__dict__.get("_nmm_ln_fold", False)), bool(module.__dict__.get("_nmm_fp32_fma", False)),
                bool(module.__dict__.get("_nmm_fp32_exact", False)))

    @staticmethod
    def _checksum(tensors):
        return float(sum(t.detach().double().abs().sum() for t in tensors.values()))

    # hooks (the spatial transformer's engine, spatial_transformer.py, overrides these three)
    def _tensors_of(self, module: nn.Module):
        return _param_tensors(module)

    def _config_of(self, module: nn.Module):
        return config_of(module)

    def _pack(self, cfg, dev_tensors, x: torch.Tensor):
        return ops.pack_params(cfg, dev_tensors, x.dtype, x.device)

    def get(self, module: nn.Module, x: torch.Tensor):
        if self.tensors is None:
            self.tensors = self._tensors_of(module)
        tensors = self.tensors
        key = self._key(x, tensors) + self._flags(module)
        if key != self.key:
            self.tensors = tensors = self._tensors_of(module)      # re-scan the tree (parameters may have been replaced)
            key = self._key(x, tensors) + self._flags(module)
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("neurons_b200: the module's parameters must be packed before CUDA-graph capture: run one forward "
                                   "outside the capture first (packing inside a capture would bake stale weights into the graph)")
            self.cfg = self._config_of(module)
            dev_tensors = {}
            for k, t in tensors.items():
                if t.device != x.device:
                    raise RuntimeError(f"neurons_b200: parameter '{k}' is on {t.device}, input on {x.device}")
                dev_tensors[k] = t.reshape(t.shape[-2:]) if k.endswith("pos_encoder.pe") else t
            self.packed = self._pack(self.cfg, dev_tensors, x)
            # once per (module, weights): wait for the packing kernels, so that the packed buffer may be used from ANY stream afterwards
            # (another stream, or a CUDA-graph capture, must not depend on un-captured work of the stream that packed)
            torch.cuda.current_stream(x.device).synchronize()
            self.key = key
            self.shape_cache.clear()
            if _WEIGHT_CHECK:
                self.checksum = self._checksum(tensors)
        else:
            if _WEIGHT_CHECK and not torch.cuda.is_current_stream_capturing():
                now = self._checksum(tensors)
                if now != self.checksum:
                    raise RuntimeError("neurons_b200 (NMM_WEIGHT_CHECK): parameters changed in place through `.data` since they were "
                                       "packed -- call neurons_b200.invalidate(model) after merging LoRA / editing weights")
        return self.cfg, self.packed


def _engine_of(module: nn.Module) -> _Engine:
    eng = module.__dict__.get("_nmm_engine")
    if eng is None:
        eng = _Engine()
        module.__dict__["_nmm_engine"] = eng      # not a submodule / buffer: invisible to state_dict()
    return eng


def motion_forward(module: nn.Module, input_tensor: torch.Tensor) -> torch.Tensor:
    """VanillaTemporalModule.forward on the B200 path.  Inference only (the reference samples under no_grad)."""
    if input_tensor.dim() != 5:
        raise AssertionError(f"Expected hidden_states to have ndim=5, but got ndim={input_tensor.dim()}.")   # :135
    if not input_tensor.is_cuda:
        raise RuntimeError("neurons_b200: the motion module runs on CUDA (sm_100) only; there is no CPU path")
    if torch.is_grad_enabled() and (input_tensor.requires_grad or any(p.requires_grad for p in module.parameters())):
        raise RuntimeError("neurons_b200: the motion-module op is inference-only; call it under torch.no_grad()")
    eng = _engine_of(module)
    cfg, packed = eng.get(module, input_tensor)
    # same computation as torch.ops.neurons_mm.forward (ops.forward_packed is its CUDA implementation), called directly with this
    # module's shape cache so the per-call host work is one dict lookup, two allocations and one C call
    if not module.__dict__.get("_nmm_carry_stats", False):
        return ops.forward_packed(input_tensor, packed, cfg, shape_cache=eng.shape_cache)
    # patch(model, carry_stats=True): the GroupNorm statistics of y ride on the output tensor to the next InflatedGroupNorm
    # (ResnetBlock3D.norm1, unet_blocks.py:407-411), and statistics riding on x are used instead of a pass over x
    B, _, F = input_tensor.shape[:3]
    y_sums = torch.empty((B * F * 32, 2), dtype=torch.float64, device=input_tensor.device)
    y = ops.forward_packed(input_tensor, packed, cfg, shape_cache=eng.shape_cache, x_sums=carried_sums(input_tensor), y_sums=y_sums)
    attach_sums(y, y_sums)
    return y


def attach_sums(t: torch.Tensor, sums: torch.Tensor) -> None:
    """Let GroupNorm statistics ride on the tensor object they describe (valid while the tensor is not modified in place)."""
    t._nmm_gn_sums = (sums, t._version, t.data_ptr(), tuple(t.shape), tuple(t.stride()))


def carried_sums(t: torch.Tensor) -> Optional[torch.Tensor]:
    rec = getattr(t, "_nmm_gn_sums", None)
    if rec is None:
        return None
    sums, version, ptr, shape, stride = rec
    if version != t._version or ptr != t.data_ptr() or shape != tuple(t.shape) or stride != tuple(t.stride()):
        return None                               # the tensor changed since the statistics were taken: recompute
    return sums


def invalidate(model: nn.Module) -> int:
    """Drop cached packed parameters (call after mutating weights in place once the model has already run)."""
    n = 0
    for m in model.modules():
        eng = m.__dict__.get("_nmm_engine")
        if eng is not None:
            eng.key = None
            eng.packed = None
            eng.tensors = None
            n += 1
    return n


def _is_motion_module(m: nn.Module) -> bool:
    return type(m).__name__ == "VanillaTemporalModule" and hasattr(m, "temporal_transformer")


def patch(model: nn.Module, carry_stats: bool = False) -> int:
    """Rebind `forward` on every VanillaTemporalModule inside `model` (reference instances included) to the CUDA op.
    Returns the number of modules patched.  Unsupported configurations raise here, never fall back silently.
    carry_stats=True: each call also emits the GroupNorm statistics of its output (from the last kernel's epilogue) and attaches
    them to the returned tensor; `patch_group_norms`-patched InflatedGroupNorms pick them up and skip their statistics pass."""
    n = 0
    for m in model.modules():
        if _is_motion_module(m):
            config_of(m)                              # raises on unsupported variants
            m.__dict__["_nmm_carry_stats"] = bool(carry_stats)

            def _fwd(self, input_tensor, temb=None, encoder_hidden_states=None, attention_mask=None, anchor_frame_idx=None):
                return motion_forward(self, input_tensor)
            m.forward = types.MethodType(_fwd, m)
            n += 1
    return n
