#!/usr/bin/env python
"""The three fp32 modes side by side on the GPU: per-call time of the spatial transformer and of the motion module in the x3 (NMM_F32X3,
default), x6 (NMM_F32X6, `_nmm_fp32_exact`) and FMA (NMM_F32, `_nmm_fp32_fma`) modes, and the x6 mode's per-kernel-class breakdown from the
library's own timers (lib.profile_begin / profile_end).  The GEMM TFLOP/s are fp32-equivalent: 2 M N K per Linear over the kernel time (an x6
GEMM issues six bf16 MMAs per product).  Shapes: the seven spatial-transformer calls of profiles/r3_spatial_fp32_attention.txt (config 2's
levels at B 2, F 8; NEURONS' 16-frame levels) and the motion module's UNet levels (B 2, F 8; the 16-frame 32 x 32 shapes).
Each figure: mean of 5 calls after 2 warm-up calls, CUDA events; run the script twice in one GPU session for the spread.  Prints the GPU's name and power limit first.  Development / profiles tool."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import neurons_b200 as nb  # noqa: E402
from neurons_b200 import lib as nlib  # noqa: E402
from oracle import motion_oracle as mo  # noqa: E402
from oracle import spatial_oracle as so  # noqa: E402

MODES = (("x3", None), ("x6", "_nmm_fp32_exact"), ("fma", "_nmm_fp32_fma"))
SPATIAL = ((320, 64, 2, 8), (640, 32, 2, 8), (1280, 16, 2, 8), (1280, 8, 2, 8), (320, 32, 2, 16), (640, 16, 2, 16), (1280, 8, 2, 16))
MOTION = ((320, 64, 2, 8), (640, 32, 2, 8), (1280, 16, 2, 8), (1280, 8, 2, 8), (320, 32, 2, 16), (640, 16, 2, 16), (1280, 8, 2, 16))


def time_call(fn, reps=5):
    for _ in range(2):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def breakdown(fn):
    nlib.profile_begin()
    fn()
    torch.cuda.synchronize()
    prof = nlib.profile_end()
    return "  ".join(f"{k} {v['total_ms']:.2f} ms ({v['flops'] / max(v['total_ms'], 1e-9) / 1e9:.1f} TF/s)" for k, v in prof.items() if v["launches"])


def spatial():
    print("# spatial transformer per call (C, side, B, F), fp32 activations; x6 breakdown from the library's timers")
    with torch.no_grad():
        for C, side, B, F in SPATIAL:
            cfg = so.SpatialConfig(C, 8, 1, 768, True)
            x = torch.randn(B, C, F, side, side, device="cuda")
            ctx = torch.randn(B, 77, 768, device="cuda")
            m = nb.Transformer3DModel(num_attention_heads=8, attention_head_dim=C // 8, in_channels=C, num_layers=1, cross_attention_dim=768,
                                      unet_use_cross_frame_attention=False, unet_use_temporal_attention=False).eval().cuda()
            ts, parts = {}, ""
            for mode, flag in MODES:
                m.__dict__.pop("_nmm_fp32_exact", None)
                m.__dict__.pop("_nmm_fp32_fma", None)
                if flag:
                    m.__dict__[flag] = True
                fn = lambda: m(x, encoder_hidden_states=ctx)  # noqa: E731
                ts[mode] = time_call(fn)
                if mode == "x6":
                    parts = breakdown(fn)
            fl = so.flops(cfg, B, F, side * side, 77)
            print(f"C={C:5d} {side:2d}x{side:<2d} B={B} F={F:2d}: " + "   ".join(f"{k} {v:7.2f} ms ({fl / v / 1e9:5.1f} TF/s)" for k, v in ts.items())
                  + f"   x6/x3 {ts['x6'] / ts['x3']:.2f}  fma/x6 {ts['fma'] / ts['x6']:.2f}   x6 breakdown: {parts}", flush=True)
            del x, m


def motion():
    print("# motion module per call (C, side, B, F), fp32 activations, 2 attention blocks + PE (the UNet's); x6 breakdown from the library's timers")
    with torch.no_grad():
        for C, side, B, F in MOTION:
            cfg = mo.MotionConfig(C, 8, 1, 2, True, 32)
            m = nb.get_motion_module(C, "Vanilla", dict(num_attention_heads=8, num_transformer_block=1, temporal_position_encoding=True,
                                                       temporal_position_encoding_max_len=32, zero_initialize=False)).eval().cuda()
            x = torch.randn(B, C, F, side, side, device="cuda")
            ts, parts = {}, ""
            for mode, flag in MODES:
                m.__dict__.pop("_nmm_fp32_exact", None)
                m.__dict__.pop("_nmm_fp32_fma", None)
                if flag:
                    m.__dict__[flag] = True
                fn = lambda: m(x, None, None)  # noqa: E731
                ts[mode] = time_call(fn)
                if mode == "x6":
                    parts = breakdown(fn)
            print(f"C={cfg.channels:5d} {side:2d}x{side:<2d} B={B} F={F:2d}: " + "   ".join(f"{k} {v:7.3f} ms" for k, v in ts.items())
                  + f"   x6/x3 {ts['x6'] / ts['x3']:.2f}  fma/x6 {ts['fma'] / ts['x6']:.2f}   x6 breakdown: {parts}", flush=True)
            del x, m


def main():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    print(f"# {name}, power limit {pl}")
    which = sys.argv[1:] or ["spatial", "motion"]
    if "spatial" in which:
        spatial()
    if "motion" in which:
        motion()


if __name__ == "__main__":
    main()
