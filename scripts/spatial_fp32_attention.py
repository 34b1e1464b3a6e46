#!/usr/bin/env python
"""fp32 spatial attention of the FMA mode (NMM_F32), measured on the GPU:
  1. the attention kernel alone, checker (NMM_OPT_SPATIAL_ATTN 31) against the tiled FMA-pipe kernel (30), over a sweep of sizes that shows
     the crossover of launch_spatial_attention's default selection; CUDA events around each call with L2 overwritten (256 MB written) before
     it (the events include the host's launch path: ~18 us is the floor of the smallest calls); fp32 TFLOP/s from the kernels' flop count,
     4 * Lq * Lkv * d_h per (image, head);
  2. per-call time of the spatial transformer in the FMA and x3 modes at config 2's four levels (B 2, F 8) and NEURONS' three (B 2, F 16),
     with the FMA mode's per-kernel-class breakdown from the library's own timers (lib.profile_begin / profile_end).
Prints the GPU's name and power limit first.  Development / profiles tool."""
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import neurons_b200 as nb  # noqa: E402
from neurons_b200 import lib as nlib  # noqa: E402
from oracle import spatial_oracle as so  # noqa: E402

CHECKER_MAX_SCORES = 3e8        # the checker beyond this takes seconds per call: not swept


def _flush(buf):
    buf.zero_()


def time_attention(variant, q, k, v, heads, flush, reps=5):
    with nlib.options({nlib.OPT_SPATIAL_ATTN: variant}):
        nb.spatial_attention(q, k, v, heads)
        ts = []
        for _ in range(reps):
            _flush(flush)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            nb.spatial_attention(q, k, v, heads)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def sweep():
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    print("# attention kernel alone: q | k | v column slices of one [images, L, 3C] fp32 buffer, 8 heads, median of 5 calls, L2 overwritten before each")
    print(f"{'dh':>4} {'L':>5} {'images':>6} {'scores':>9} {'checker ms':>11} {'tiled ms':>9} {'chk TF/s':>9} {'tiled TF/s':>10} {'faster':>8}")
    for dh in (40, 80, 160):
        C = 8 * dh
        for L in (32, 64, 128, 256, 512, 1024, 2048, 4096):
            for images in (1, 2, 4, 16):
                scores = float(L) * L * images * 8
                qkv = torch.randn(images, L, 3 * C, device="cuda")
                q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
                fl = 4.0 * scores * dh
                tc = time_attention(31, q, k, v, 8, flush) if scores <= CHECKER_MAX_SCORES else float("nan")
                tt = time_attention(30, q, k, v, 8, flush)
                faster = "-" if tc != tc else ("tiled" if tt < tc else "checker")
                print(f"{dh:>4} {L:>5} {images:>6} {scores:>9.2e} {tc:>11.4f} {tt:>9.4f} {fl / tc / 1e9:>9.2f} {fl / tt / 1e9:>10.2f} {faster:>8}", flush=True)
                del qkv


def build(cfg, fma):
    m = nb.Transformer3DModel(num_attention_heads=cfg.heads, attention_head_dim=cfg.head_dim, in_channels=cfg.channels, num_layers=cfg.layers,
                              cross_attention_dim=cfg.ctx_dim, use_linear_projection=not cfg.conv_proj, unet_use_cross_frame_attention=False,
                              unet_use_temporal_attention=False).eval().cuda()
    if fma:
        m.__dict__["_nmm_fp32_fma"] = True
    return m


def modules():
    print("# spatial transformer per call (C, side, B, F), fp32 activations; mean of 5 calls after 2 warm-up; FMA-mode breakdown from the library's timers")
    with torch.no_grad():
        for C, side, B, F in ((320, 64, 2, 8), (640, 32, 2, 8), (1280, 16, 2, 8), (1280, 8, 2, 8), (320, 32, 2, 16), (640, 16, 2, 16), (1280, 8, 2, 16)):
            cfg = so.SpatialConfig(C, 8, 1, 768, True)
            x = torch.randn(B, C, F, side, side, device="cuda")
            ctx = torch.randn(B, 77, 768, device="cuda")
            ts = []
            for fma in (False, True):
                m = build(cfg, fma)
                for _ in range(2):
                    m(x, encoder_hidden_states=ctx)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    m(x, encoder_hidden_states=ctx)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / 5)
            nlib.profile_begin()
            m(x, encoder_hidden_states=ctx)
            torch.cuda.synchronize()
            prof = nlib.profile_end()
            fl = so.flops(cfg, B, F, side * side, 77)
            parts = "  ".join(f"{k} {v['total_ms']:.2f} ms ({v['flops'] / max(v['total_ms'], 1e-9) / 1e9:.1f} TF/s)" for k, v in prof.items() if v["launches"])
            print(f"C={C:5d} {side:2d}x{side:<2d} B={B} F={F:2d}: x3 {ts[0]:7.2f} ms ({fl / ts[0] / 1e9:5.1f} TF/s)   fma {ts[1]:7.2f} ms "
                  f"({fl / ts[1] / 1e9:5.1f} TF/s)   fma breakdown: {parts}", flush=True)
            del x, m


def main():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    print(f"# {name}, power limit {pl}")
    which = sys.argv[1:] or ["sweep", "modules"]
    if "sweep" in which:
        sweep()
    if "modules" in which:
        modules()


if __name__ == "__main__":
    main()
