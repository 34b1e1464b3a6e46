#!/usr/bin/env python
"""fp32 modes of the spatial transformer (SURVEY 8(f) N3): accuracy against the reference-generated fixtures and time per call at the UNet levels,
NMM_F32X3 (Linears AND attention on the tensor cores, 3 bf16 MMAs per product) vs NMM_F32 (FMA-pipe GEMM + fp32 FMA-pipe attention)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import neurons_b200 as nb  # noqa: E402
from tests.test_spatial_oracle import load_sp_golden, sp_golden_names  # noqa: E402


def build(cfg, params, fma):
    m = nb.Transformer3DModel(num_attention_heads=cfg.heads, attention_head_dim=cfg.head_dim, in_channels=cfg.channels, num_layers=cfg.layers,
                              cross_attention_dim=cfg.ctx_dim, use_linear_projection=not cfg.conv_proj, unet_use_cross_frame_attention=False,
                              unet_use_temporal_attention=False)
    if params is not None:
        m.load_state_dict(params, strict=True)
    m = m.eval().cuda()
    if fma:
        m.__dict__["_nmm_fp32_fma"] = True
    return m


def main():
    with torch.no_grad():
        for name in sp_golden_names():
            fx, cfg, params, x, ctx = load_sp_golden(name)
            errs = []
            for fma in (False, True):
                y = build(cfg, params, fma)(x.cuda(), encoder_hidden_states=ctx.cuda()).sample
                errs.append((y.cpu() - fx["out_ref_fp32"]).abs().max().item())
            print(f"{name:26s} max-abs vs reference fp32: x3 {errs[0]:.2e}   fma {errs[1]:.2e}   (bar 1e-4)", flush=True)
        from oracle import spatial_oracle as so
        for C, side in ((320, 64), (640, 32), (1280, 16), (1280, 8)):
            cfg = so.SpatialConfig(C, 8, 1, 768, True)
            x = torch.randn(2, C, 8, side, side, device="cuda")
            ctx = torch.randn(2, 77, 768, device="cuda")
            ts = []
            for fma in (False, True):
                m = build(cfg, None, fma)
                for _ in range(2):
                    m(x, encoder_hidden_states=ctx)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    m(x, encoder_hidden_states=ctx)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / 5)
            fl = so.flops(cfg, 2, 8, side * side, 77)
            print(f"fp32 C={C:5d} {side:2d}x{side:<2d}: x3 {ts[0]:7.2f} ms ({fl / ts[0] / 1e9:6.1f} TF/s)   fma {ts[1]:7.2f} ms ({fl / ts[1] / 1e9:6.1f} TF/s)", flush=True)


if __name__ == "__main__":
    main()
